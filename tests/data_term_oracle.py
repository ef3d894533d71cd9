"""Numpy reference for the Chambolle-Pock iteration with the L1 and weighted-L2 data terms.  TEST INFRASTRUCTURE ONLY.

Written in the style of oracle.tv_oracle.cp_rof_step and built only from that module's operators (D, D_T, the projection,
L21), independently of the CUDA code.  It lives here rather than in oracle/tv_oracle.py so that the pinned oracle module,
checked against the reference's goldens, stays unchanged.
"""
import numpy as np

from oracle import tv_oracle as orc


def cp_data_step(x, xbar, x0, y, data_term="l2", data_weight=None, scheme="hybrid", lam=0.1, sigma=0.5, tau=1.0 / 13.0, theta=1.0,
                 **weights):
    """cp_rof_step with another data term F(x) = sum_v w_v phi(x_v - x0_v): phi = 0.5 r^2 ("l2") or |r| ("l1"); w = data_weight
    (broadcast to the image, >= 0), or 1 when None.  Only the prox of the primal step changes; with v = x - tau D^T y:
        l2: x_new = (v + tau w x0) / (1 + tau w)
        l1: x_new = x0 + sign(v - x0) max(|v - x0| - tau w, 0)      (Chambolle & Pock 2011, Sec. 6.2.2)
    Returns (x, xbar, y, primal_energy) with primal_energy = F(x_new) + lam*L21(D xbar_old).  tau w and 1 + tau w are
    formed in float64 and rounded once, so that "l2" with w = 1 is cp_rof_step bit for bit."""
    if data_term not in ("l2", "l1"):
        raise ValueError("data_term must be 'l2' or 'l1'")
    dt = x.dtype.type
    w64 = np.ones(x.shape) if data_weight is None else np.broadcast_to(np.asarray(data_weight, dtype=np.float64), x.shape)
    tw = (tau * w64).astype(x.dtype)
    Dxb = orc.D(xbar, scheme, **weights)
    y = orc.project_l2_ball(y + dt(sigma) * Dxb, lam)
    v = x - dt(tau) * orc.D_T(y, scheme, **weights)
    if data_term == "l2":
        x_new = (v + tw * x0) / (1.0 + tau * w64).astype(x.dtype)
        fid = 0.5 * np.sum(w64 * np.square(x_new - x0), dtype=np.float64)
    else:
        d = v - x0
        x_new = x0 + np.sign(d) * np.maximum(np.abs(d) - tw, dt(0))
        fid = np.sum(w64 * np.abs(x_new - x0), dtype=np.float64)
    xbar = x_new + dt(theta) * (x_new - x)
    energy = fid + lam * np.float64(orc.l21(Dxb))
    return x_new, xbar, y, float(energy)


def primal_energy(x, x0, data_term, data_weight, scheme, lam, **weights):
    """F(x) + lam TV(x)."""
    w64 = np.ones(x.shape) if data_weight is None else np.broadcast_to(np.asarray(data_weight, dtype=np.float64), x.shape)
    r = (x - x0).astype(np.float64)
    fid = 0.5 * np.sum(w64 * r * r) if data_term == "l2" else np.sum(w64 * np.abs(r))
    return float(fid + lam * orc.l21(orc.D(x, scheme, **weights)))


def dual_energy(y, x0, data_term, data_weight, scheme, **weights):
    """Dual objective at a feasible y (|y_v| <= lam), s = D^T y, all w > 0:
        l2: sum_v (s x0 - s^2 / (2 w))
        l1: c <s, x0> with c = min(1, min_v w_v / |s_v|) (y scaled into the box |s_v| <= w_v of the conjugate)."""
    s = orc.D_T(y, scheme, **weights).astype(np.float64)
    w64 = np.ones(s.shape) if data_weight is None else np.broadcast_to(np.asarray(data_weight, dtype=np.float64), s.shape)
    x0 = x0.astype(np.float64)
    if data_term == "l2":
        return float(np.sum(s * x0 - s * s / (2.0 * w64)))
    a = np.abs(s)
    c = min(1.0, float(np.min(np.where(a > 0, w64 / np.where(a > 0, a, 1.0), np.inf))))
    return float(c * np.sum(s * x0))


def run(x0, n_iter, data_term="l2", data_weight=None, scheme="hybrid", lam=0.1, sigma=0.5, tau=None, theta=1.0, **weights):
    """n_iter iterations from x = xbar = x0, y = 0; returns (x, xbar, y, energy of the last iteration)."""
    Nz, M = x0.shape[:2]
    Nd = orc.num_components(scheme, Nz, M, weights.get("reg_z_over_reg", 1.0), weights.get("reg_time", 0.0))
    x, xb, y = x0.copy(), x0.copy(), np.zeros((Nz, Nd) + x0.shape[1:], dtype=x0.dtype)
    e = None
    for _ in range(n_iter):
        x, xb, y, e = cp_data_step(x, xb, x0, y, data_term, data_weight, scheme, lam=lam, sigma=sigma, tau=tau, theta=theta, **weights)
    return x, xb, y, e
