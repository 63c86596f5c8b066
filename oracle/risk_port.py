"""numpy twin of the risk-averse backups (nested mean-CVaR, include/sdp_b200.h SdpRisk).

TEST INFRASTRUCTURE ONLY - the reference of tests/test_risk.py.  The reference has no risk
measure; this restates the arithmetic contract of the kernels with explicit loops over the
nodes (no np.inner, whose summation order is BLAS's), so that it gives the kernels' bits:

  E   = ((0 + v_0*p_0) + v_1*p_1) + ...                   nodes in w order
  C   = NaN if any v_w is NaN; else the walk over the nodes sorted by v descending (stable
        argsort of -v: ties keep the lower w first, -0 == +0) of the upper tail of mass beta
  rho = E*w_mean + C*w_cvar

`PortSolver` is the oracle port (oracle/ref_port.py) with that backup in value iteration, the
recursion and policy evaluation.
"""
import numpy as np

from . import ref_port

__all__ = ["risk_constants", "risk_values", "PortSolver", "port_api"]


def risk_constants(alpha, weight):
    """(inv_beta, beta, w_mean, w_cvar), computed in fp64 as the host does"""
    beta = 1.0 - float(alpha)
    return 1.0 / beta, beta, 1.0 - float(weight), float(weight)


def risk_values(V, p, consts):
    """rho of every row of V [n, W] (node values) under probabilities p [W]"""
    inv_beta, beta, w_mean, w_cvar = consts
    V = np.asarray(V, dtype=np.float64)
    p = np.asarray(p, dtype=np.float64)
    n, W = V.shape
    with np.errstate(invalid="ignore", over="ignore"):
        E = np.zeros(n)
        for w in range(W):
            E = E + V[:, w] * p[w]
        order = np.argsort(-V, axis=1, kind="stable")
        rows = np.arange(n)
        cum = np.zeros(n)
        acc = np.zeros(n)
        done = np.zeros(n, dtype=bool)
        for k in range(W):
            idx = order[:, k]
            pk = p[idx]
            vk = V[rows, idx]
            live = ~done & (pk != 0.0)
            stop = live & (cum >= beta)
            done |= stop
            live &= ~stop
            r = beta - cum
            full = live & (pk <= r)
            part = live & ~full
            acc = np.where(full, acc + vk * pk, acc)
            cum = np.where(full, cum + pk, cum)
            acc = np.where(part, acc + vk * r, acc)
            done |= part
        C = acc * inv_beta
        C[np.isnan(V).any(axis=1)] = np.nan
        return E * w_mean + C * w_cvar


class PortSolver(ref_port.PortSolver):
    """the oracle port with the risk backup; `risk` = (alpha, weight), or None for the port's own
    (np.inner) expectation"""

    def __init__(self, sys, interp="c", risk=None):
        super().__init__(sys, interp)
        self.risk = risk

    def value_at_state(self, x_k, J_interp, t_k=None, want_index=False):
        if self.risk is None or len(self.perturb_grid) == 0:
            return super().value_at_state(x_k, J_interp, t_k, want_index)
        u_grids, control_dims = self.control_grids(x_k, t_k)
        nc = len(u_grids)
        m = len(self.perturb_grid)
        for i in range(nc):
            u_grids[i].shape = (1,) * i + (-1,) + (1,) * (nc - 1 - i + m)
        w_args, w_shape, p = self._perturb_product()
        args = x_k + tuple(u_grids) + w_args
        if t_k is not None:
            args = (t_k,) + args
        x_next = self.sys.dyn(*args, **self.sys.params)
        g = self.sys.cost(*args, **self.sys.params)
        J_grid = g + J_interp(*x_next)
        V = np.broadcast_to(J_grid, control_dims + w_shape).reshape(-1, len(p))
        J = risk_values(V, p, risk_constants(*self.risk)).reshape(control_dims)
        flat = J.argmin()
        ind = np.unravel_index(flat, control_dims)
        u_opt = [u_grids[i].flatten()[ind[i]] for i in range(nc)]
        if want_index:
            return J[ind], u_opt, int(flat), J
        return J[ind], u_opt

    def eval_policy(self, pol, n_iter, rel_dp=False, J_zero=None, report_time=False, J_ref_full=False):
        if self.risk is None:
            return super().eval_policy(pol, n_iter, rel_dp, J_zero, report_time, J_ref_full)
        dims = self._state_grid_shape
        ns = len(self.sys.state)
        J_pol = np.zeros(dims) if J_zero is None else J_zero
        J_ref = np.zeros(n_iter)
        ref_ind = self._state_ref_ind
        nc = len(self.sys.control)
        m = len(self.perturb_grid)
        w_args, w_shape, p = self._perturb_product()
        sg = tuple(np.reshape(self.state_grid[i], (1,) * i + (-1,) + (1,) * (ns - 1 - i + m))
                   for i in range(ns))
        consts = risk_constants(*self.risk)
        for k in range(n_iter):
            J_interp = self.interp_on_state(J_pol)
            u_k = [pol[..., i].reshape(dims + (1,) * m) for i in range(nc)]
            args = sg + tuple(u_k) + w_args
            x_next = self.sys.dyn(*args, **self.sys.params)
            g = self.sys.cost(*args, **self.sys.params)
            J_grid = g + J_interp(*x_next)
            V = np.broadcast_to(J_grid, dims + w_shape).reshape(-1, len(p))
            J_pol = risk_values(V, p, consts).reshape(dims)
            if rel_dp:
                J_ref[k] = J_pol[ref_ind]
                J_pol = J_pol - J_ref[k]
        if rel_dp:
            return J_pol, (J_ref if J_ref_full else J_ref[-1])
        return J_pol

    def value_iteration_states(self, J_next, states):
        """(J, flat argmin) of the given flat state indices only (sampled checks of large grids)"""
        dims = tuple(len(g) for g in self.state_grid)
        J_interp = self.interp_on_state(J_next)
        J = np.zeros(len(states))
        idx = np.zeros(len(states), dtype=np.int64)
        for j, s in enumerate(states):
            ind_x = np.unravel_index(int(s), dims)
            x_k = tuple(g[i] for g, i in zip(self.state_grid, ind_x))
            J[j], _, idx[j], _ = self.value_at_state(x_k, J_interp, None, True)
        return J, idx


class _PortAPI(ref_port._PortAPI):
    def __init__(self, risk, interp="c"):
        super().__init__(interp)
        self._risk = risk

    def DPSolver(self, sys, **kw):
        return PortSolver(sys, interp=self._interp, risk=self._risk)


def port_api(risk, interp="c"):
    """`api` object for the tests/workloads.py factories: port solvers with the risk backup
    `risk` = (alpha, weight)"""
    return _PortAPI(risk, interp)

