"""Float64 numpy model of the condensed QP the CUDA kernels build and solve (TEST INFRASTRUCTURE ONLY).

The reference hands cvxpy the sparse (x, u) problem (main/lib/mpc.py:151-196).  Because the steering
operating point is always 0 (`dref == 0`, mpc.py:96) the linearised dynamics decouple into

    v_t   = v0   + dt   * sum_{k<t} a_k
    psi_t = psi0 + sum_{k<t} g_k * delta_k                       g_k = dt * vbar_k / L
    X_t   = X0 + sum_{j<t} [ alpha_j v_j - beta_j (psi_j - phibar_j) ]    alpha = dt cos(phibar), beta = dt vbar sin(phibar)
    Y_t   = Y0 + sum_{j<t} [ gamma_j v_j + kappa_j (psi_j - phibar_j) ]   gamma = dt sin(phibar), kappa = dt vbar cos(phibar)

so the states are eliminated exactly: n = 2T unknowns u = [a_0..a_{T-1}, delta_0..delta_{T-1}] and
m = 4T-1 two-sided rows (T accel boxes, T steer boxes, T-1 steer-rate rows, T speed rows as bounds on the
running sum of a).  This file exists to localise a discrepancy (condensing vs solver) and to prototype the
solver; tests compare it with the sparse oracle.

Since the second half of round 2 the CUDA kernel solves the same problem in the unknowns [s_0..s_{T-1}, delta] with
s_k = a_0 + ... + a_k (a linear change of variables: same rows, same slacks, same interior-point iterates): the
speed rows become boxes on s_k, the acceleration rows differences, and A' W A is tridiagonal in both blocks.
`condense_cumulative` below is the numpy statement of that condensing; the solver model further down is still
written in the a_k form.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from .mpc_oracle import Params, stage_state_weight


@dataclass
class CondensedQP:
    P: np.ndarray       # (n, n)   1/2 u'Pu + q'u + c0
    q: np.ndarray
    c0: float
    A: np.ndarray       # (m, n) constraint rows (constant for a given T)
    lo: np.ndarray      # (m,)
    hi: np.ndarray
    S: np.ndarray       # (T+1, 4, n)  state sensitivities: x_t = x_t^free + S_t u
    xfree: np.ndarray   # (T+1, 4)


def constraint_matrix(T: int) -> np.ndarray:
    n = 2 * T
    A = np.zeros((4 * T - 1, n))
    A[:n, :n] = np.eye(n)
    for k in range(T - 1):
        A[n + k, T + k] = -1.0
        A[n + k, T + k + 1] = 1.0
    for t in range(1, T + 1):
        A[3 * T - 1 + (t - 1), :t] = 1.0          # running sum of a (speed rows, scaled by 1/dt in the bounds)
    return A


def condense(p: Params, xref: np.ndarray, xbar: np.ndarray, x0, reaches_end) -> CondensedQP:
    T, dt = p.T, p.dt
    n = 2 * T
    vb, ph = xbar[2], xbar[3]
    alpha = dt * np.cos(ph[:T])
    beta = dt * vb[:T] * np.sin(ph[:T])
    gamma = dt * np.sin(ph[:T])
    kappa = dt * vb[:T] * np.cos(ph[:T])
    g = dt * vb[:T] / p.L
    S = np.zeros((T + 1, 4, n))
    xfree = np.zeros((T + 1, 4))
    xfree[0] = x0
    for t in range(T):
        X, Y, v, psi = xfree[t]
        xfree[t + 1] = (X + alpha[t] * v - beta[t] * (psi - ph[t]), Y + gamma[t] * v + kappa[t] * (psi - ph[t]), v, psi)
        S[t + 1, 0] = S[t, 0] + alpha[t] * S[t, 2] - beta[t] * S[t, 3]
        S[t + 1, 1] = S[t, 1] + gamma[t] * S[t, 2] + kappa[t] * S[t, 3]
        S[t + 1, 2] = S[t, 2]
        S[t + 1, 3] = S[t, 3]
        S[t + 1, 2, t] += dt
        S[t + 1, 3, T + t] += g[t]
    P = np.zeros((n, n))
    q = np.zeros(n)
    c0 = 0.0
    for t in range(1, T + 1):
        Q = stage_state_weight(p, float(xref[3, t]), bool(reaches_end[t]))
        e = xfree[t] - xref[:, t]
        P += 2.0 * S[t].T @ Q @ S[t]
        q += 2.0 * S[t].T @ (Q @ e)
        c0 += float(e @ Q @ e)
    for t in range(T):
        r = p.R_end if reaches_end[t] else p.R
        P[t, t] += 2.0 * r[0]
        P[T + t, T + t] += 2.0 * r[1]
    for t in range(T - 1):
        for blk, w in ((0, p.Rd[0]), (T, p.Rd[1])):
            i, j = blk + t, blk + t + 1
            P[i, i] += 2.0 * w
            P[j, j] += 2.0 * w
            P[i, j] -= 2.0 * w
            P[j, i] -= 2.0 * w
    A = constraint_matrix(T)
    lim = p.max_dsteer * dt
    lo = np.concatenate([np.full(T, p.max_decel), np.full(T, -p.max_steer), np.full(T - 1, -lim),
                         np.full(T, (p.min_speed - x0[2]) / dt)])
    hi = np.concatenate([np.full(T, p.max_accel), np.full(T, p.max_steer), np.full(T - 1, lim),
                         np.full(T, (p.speed - x0[2]) / dt)])
    return CondensedQP(P=P, q=q, c0=c0, A=A, lo=lo, hi=hi, S=S, xfree=xfree)


# ----------------------------------------------------------------------------------------------------
# The same problem in cumulative accelerations (what csrc/jmpc_step.cuh builds): speed rows are boxes on s_k,
# acceleration rows differences, A' W A tridiagonal in both blocks.
# ----------------------------------------------------------------------------------------------------
def cumulative_transform(T: int) -> np.ndarray:
    """E with [a; delta] = E [s; delta]:  a_k = s_k - s_{k-1}."""
    D = np.eye(T) - np.eye(T, k=-1)
    return np.block([[D, np.zeros((T, T))], [np.zeros((T, T)), np.eye(T)]])


def _sfx(v):
    return np.cumsum(v[::-1])[::-1]


def condense_cumulative(p: Params, xref: np.ndarray, xbar: np.ndarray, x0, reach):
    """(P, q) of the condensed QP in the unknowns the CUDA kernel uses since round 2: [s_0..s_{T-1}, delta_0..delta_{T-1}]
    with s_k = a_0 + ... + a_k, computed the way the kernel computes it (suffix sums of the stage weights and of
    their first / second moments).  Must equal E' P E, E' q of `condense` with u = E [s; delta], a_k = s_k - s_{k-1}."""
    T, dt = p.T, p.dt
    vb, ph = xbar[2], xbar[3]
    al = np.append(dt * np.cos(ph[:T]), 0.0)            # index T: 0 (s_{T-1} moves no position)
    be = dt * vb[:T] * np.sin(ph[:T])
    ga = np.append(dt * np.sin(ph[:T]), 0.0)
    ka = dt * vb[:T] * np.cos(ph[:T])
    g = dt * vb[:T] / p.L
    cb = np.concatenate([[0.0], np.cumsum(be)])          # exclusive prefix sums, t = 0..T
    ck = np.concatenate([[0.0], np.cumsum(ka)])
    cb -= cb[T // 2]; ck -= ck[T // 2]                   # centred as in the kernel
    W = np.zeros((T + 2, 4, 4))
    for t in range(1, T + 1):
        W[t] = stage_state_weight(p, float(xref[3, t]), bool(reach[t]))
    w11, w12, w22, wv, wpsi = W[:, 0, 0], W[:, 0, 1], W[:, 1, 1], W[:, 2, 2], W[:, 3, 3]
    # free response (s = 0, delta = 0)
    xf = np.zeros(T + 1); yf = np.zeros(T + 1)
    xf[0], yf[0] = x0[0], x0[1]
    for t in range(T):
        xf[t + 1] = xf[t] + al[t] * x0[2] - be[t] * (x0[3] - ph[t])
        yf[t + 1] = yf[t] + ga[t] * x0[2] + ka[t] * (x0[3] - ph[t])
    ex = np.append(xf - xref[0], 0.0); ey = np.append(yf - xref[1], 0.0)
    ev = np.append(x0[2] - xref[2], 0.0); eps = np.append(x0[3] - xref[3], 0.0)
    WeX, WeY = w11 * ex + w12 * ey, w12 * ex + w22 * ey
    # suffix sums over stages t >= m, m = 0..T+1 (index T+1: 0)
    B_, K_ = np.append(cb, 0.0), np.append(ck, 0.0)
    S11, S12, S22 = _sfx(w11), _sfx(w12), _sfx(w22)
    M11B, M12B, M12K, M22K = _sfx(w11 * B_), _sfx(w12 * B_), _sfx(w12 * K_), _sfx(w22 * K_)
    M11BB, M12BK, M22KK = _sfx(w11 * B_ * B_), _sfx(w12 * B_ * K_), _sfx(w22 * K_ * K_)
    SPSI, SX, SY, SE = _sfx(wpsi), _sfx(WeX), _sfx(WeY), _sfx(wpsi * eps)
    SXB, SYK = _sfx(WeX * B_), _sfx(WeY * K_)
    n = 2 * T
    P = np.zeros((n, n)); q = np.zeros(n)
    dt2 = dt * dt
    for i in range(T):
        for j in range(i + 1):
            m = min(i + 2, T + 1)                        # max(i, j) + 2
            P[i, j] = 2 * dt2 * (al[i + 1] * al[j + 1] * S11[m] + (al[i + 1] * ga[j + 1] + ga[i + 1] * al[j + 1]) * S12[m]
                                 + ga[i + 1] * ga[j + 1] * S22[m])
        P[i, i] += 2 * dt2 * wv[i + 1]
        m = min(i + 2, T + 1)
        q[i] = 2 * dt * (al[i + 1] * SX[m] + ga[i + 1] * SY[m]) + 2 * dt * wv[i + 1] * ev[i + 1]
    # input weights on a = D s: B = D' M D with the tridiagonal M of the a-formulation
    def Mw(i, j):
        if i >= T or j >= T or abs(i - j) > 1:
            return 0.0
        if i == j:
            r = (p.R_end if reach[i] else p.R)[0]
            nbr = (1 if (i == 0 or i == T - 1) else 2) if T >= 2 else 0
            return 2 * r + 2 * p.Rd[0] * nbr
        return -2 * p.Rd[0]
    for i in range(T):
        for j in range(max(0, i - 2), i + 1):
            P[i, j] += Mw(i, j) - Mw(i + 1, j) - Mw(i, j + 1) + Mw(i + 1, j + 1)
    for i in range(T):                                   # steer (row) x cumulative acceleration (col)
        for j in range(T):
            m = min(max(i + 1, j + 2), T + 1)
            bi, ki = cb[i + 1], ck[i + 1]
            acc = (-al[j + 1] * (M11B[m] - bi * S11[m]) - ga[j + 1] * (M12B[m] - bi * S12[m])
                   + al[j + 1] * (M12K[m] - ki * S12[m]) + ga[j + 1] * (M22K[m] - ki * S22[m]))
            P[T + i, j] = 2 * g[i] * dt * acc
    for i in range(T):                                   # steer x steer, as in the a-formulation
        for j in range(i + 1):
            m = i + 1
            bi, ki, bj, kj = cb[i + 1], ck[i + 1], cb[j + 1], ck[j + 1]
            s11 = M11BB[m] - (bi + bj) * M11B[m] + bi * bj * S11[m]
            s12a = M12BK[m] - kj * M12B[m] - bi * M12K[m] + bi * kj * S12[m]
            s12b = M12BK[m] - bj * M12K[m] - ki * M12B[m] + ki * bj * S12[m]
            s22 = M22KK[m] - (ki + kj) * M22K[m] + ki * kj * S22[m]
            P[T + i, T + j] = 2 * g[i] * g[j] * (s11 - s12a - s12b + s22 + SPSI[m])
        r = (p.R_end if reach[i] else p.R)[1]
        nbr = (1 if (i == 0 or i == T - 1) else 2) if T >= 2 else 0
        P[T + i, T + i] += 2 * r + 2 * p.Rd[1] * nbr
        if i >= 1:
            P[T + i, T + i - 1] -= 2 * p.Rd[1]
        m = i + 1
        q[T + i] = 2 * g[i] * (-(SXB[m] - cb[i + 1] * SX[m]) + (SYK[m] - ck[i + 1] * SY[m]) + SE[m])
    P = np.tril(P) + np.tril(P, -1).T
    return P, q


def states_from_controls(c: CondensedQP, u: np.ndarray) -> np.ndarray:
    """(4, T+1) predicted states [x, y, v, yaw] of the linearised model for controls u."""
    return (c.xfree + c.S @ u).T


def objective(c: CondensedQP, u: np.ndarray) -> float:
    return float(0.5 * u @ c.P @ u + c.q @ u + c.c0)


# ----------------------------------------------------------------------------------------------------
# Model of the solver the CUDA kernel runs: Mehrotra predictor-corrector on the condensed QP with the
# constraint rows grouped per stage k (accel box, steer box, steer-rate row k -> k+1, speed row t = k+1).
# K = P + A' diag(w) A is assembled from that structure exactly as the kernel does it.
# ----------------------------------------------------------------------------------------------------
def _rows_apply(T, u):
    """A u, as four per-stage vectors (abox, dbox, rate, speed-sum)."""
    a, d = u[:T], u[T:]
    rate = np.zeros(T)
    rate[:T - 1] = d[1:] - d[:-1]
    return np.stack([a, d, rate, np.cumsum(a)])


def _rows_apply_T(T, t):
    """A' t for per-stage row values t[4, T] (rate row T-1 does not exist and must be 0)."""
    out = np.zeros(2 * T)
    out[:T] = t[0] + np.cumsum(t[3][::-1])[::-1]
    out[T:] = t[1]
    out[T:2 * T - 1] -= t[2][:T - 1]
    out[T + 1:] += t[2][:T - 1]
    return out


def _assemble_K(T, P, w):
    K = P.copy()
    idx = np.arange(T)
    K[idx, idx] += w[0]
    K[T + idx, T + idx] += w[1]
    for k in range(T - 1):
        K[T + k, T + k] += w[2][k]
        K[T + k + 1, T + k + 1] += w[2][k]
        K[T + k, T + k + 1] -= w[2][k]
        K[T + k + 1, T + k] -= w[2][k]
    suffix = np.cumsum(w[3][::-1])[::-1]               # suffix[i] = sum_{k >= i} w_speed[k]
    K[:T, :T] += suffix[np.maximum.outer(idx, idx)]
    return K


# the same three structure functions in the unknowns [s; delta] of the CUDA kernel (s_k = a_0 + ... + a_k): the
# acceleration row is s_k - s_{k-1}, the speed row s_k itself, and A' W A is tridiagonal in both blocks
def _rows_apply_cum(T, u):
    s, d = u[:T], u[T:]
    rate = np.zeros(T)
    rate[:T - 1] = d[1:] - d[:-1]
    return np.stack([s - np.concatenate([[0.0], s[:-1]]), d, rate, s])


def _rows_apply_T_cum(T, t):
    out = np.zeros(2 * T)
    out[:T] = t[0] - np.append(t[0][1:], 0.0) + t[3]
    out[T:] = t[1]
    out[T:2 * T - 1] -= t[2][:T - 1]
    out[T + 1:] += t[2][:T - 1]
    return out


def _assemble_K_cum(T, P, w):
    K = P.copy()
    idx = np.arange(T)
    K[idx, idx] += w[0] + np.append(w[0][1:], 0.0) + w[3]
    K[T + idx, T + idx] += w[1]
    for k in range(1, T):
        K[k, k - 1] -= w[0][k]
        K[k - 1, k] -= w[0][k]
    for k in range(T - 1):
        K[T + k, T + k] += w[2][k]
        K[T + k + 1, T + k + 1] += w[2][k]
        K[T + k, T + k + 1] -= w[2][k]
        K[T + k + 1, T + k] -= w[2][k]
    return K


def ipm_solve(c: CondensedQP, max_iter: int = 40, mu_tol: float = 1e-13, s_min: float = 1e-2, lam0: float = 1.0,
              cumulative: bool = False):
    """Returns (u, iterations, converged) of `ipm_solve_exit` with the kernel's default tolerances."""
    return ipm_solve_exit(c, max_iter=max_iter, mu_tol=mu_tol, s_min=s_min, lam0=lam0, cumulative=cumulative)[:3]


def ipm_solve_exit(c: CondensedQP, max_iter: int = 40, mu_tol: float = 1e-13, s_min: float = 1e-2, lam0: float = 1.0,
                   cumulative: bool = False, tol_res: float = 1e-9, init_mu: float = 0.0):
    """Returns (u, iterations, converged, exit).  `cumulative`: iterate in the kernel's unknowns [s; delta] (c.P, c.q must
    then be the Hessian / linear term in those unknowns); the result is still returned as controls [a; delta].

    The exits are those of step_solve in csrc/jmpc_step.cuh, tested in the same order on the same quantities:

      "strict"           mu <= mu_tol, every primal row <= tol_res, dual residual <= tol_res * gscale;
      "complementarity"  mu <= 1e-3 mu_tol with the primal rows strict;
      "reduced"          the iteration cap, with the last iterate tested inside mu <= 1e-9, rows <= 1e-7 and
                         dual <= 1e-7 gscale (accepted: the kernel reports the solve as converged);
      "breakdown"        the factorisation fails (a non-positive pivot in the kernel, numpy's cholesky raising here) on
                         an iterate with mu <= 1e-11, rows and dual <= 1e-9 (times gscale);
      "cap"              the iteration cap without the reduced tolerances (a failed solve);
      "diverged"         the factorisation fails anywhere else: the kernel patches the pivot and carries on, which this
                         model cannot follow (a failed solve here, whatever the kernel makes of it).

    gscale = 1 + max |q|.  `iterations` counts the completed Newton steps, as the kernel's `iters` output does.
    `init_mu > 0` starts the multipliers centred at init_mu / s, as the kernel does; otherwise at `lam0`."""
    T = len(c.q) // 2
    n = 2 * T
    _rows_apply, _rows_apply_T, _assemble_K = ((_rows_apply_cum, _rows_apply_T_cum, _assemble_K_cum) if cumulative else
                                               (globals()["_rows_apply"], globals()["_rows_apply_T"], globals()["_assemble_K"]))
    hi = np.stack([c.hi[:T], c.hi[T:2 * T], np.append(c.hi[2 * T:3 * T - 1], 1.0), c.hi[3 * T - 1:]])
    lo = np.stack([c.lo[:T], c.lo[T:2 * T], np.append(c.lo[2 * T:3 * T - 1], -1.0), c.lo[3 * T - 1:]])
    live = np.ones((4, T), bool)
    live[2, T - 1] = False                                   # there is no rate row for the last stage
    nrow = 2 * live.sum()
    u = np.zeros(n)
    z = _rows_apply(T, u)
    sh = np.maximum(hi - z, s_min)
    sl = np.maximum(z - lo, s_min)
    if init_mu > 0.0:
        lh = np.where(live, init_mu / sh, 0.0)
        ll = np.where(live, init_mu / sl, 0.0)
    else:
        lh = np.where(live, lam0, 0.0)
        ll = np.where(live, lam0, 0.0)
    gscale = 1.0 + np.abs(c.q).max()

    def result(it, ok, kind):
        return (cumulative_transform(T) @ u if cumulative else u), it, ok, kind

    acceptable = False
    for it in range(max_iter):
        z = _rows_apply(T, u)
        rd = c.P @ u + c.q + _rows_apply_T(T, np.where(live, lh - ll, 0.0))
        rph = np.where(live, z + sh - hi, 0.0)
        rpl = np.where(live, -z + sl + lo, 0.0)
        mu = float((lh * sh + ll * sl)[live].sum()) / nrow
        rp = max(np.abs(rph).max(), np.abs(rpl).max())
        rdm = np.abs(rd).max()
        if mu <= mu_tol and rp <= tol_res and rdm <= tol_res * gscale:
            return result(it, True, "strict")
        if mu <= 1e-3 * mu_tol and rp <= tol_res:
            return result(it, True, "complementarity")
        acceptable = mu <= 1e-9 and rp <= 1e-7 and rdm <= 1e-7 * gscale
        w = np.where(live, lh / sh + ll / sl, 0.0)
        K = _assemble_K(T, c.P, w)
        try:
            Lc = np.linalg.cholesky(K)
        except np.linalg.LinAlgError:
            if mu <= 1e-11 and rp <= 1e-9 and rdm <= 1e-9 * gscale:
                return result(it, True, "breakdown")
            return result(it, False, "diverged")

        def newton(rch, rcl):
            th = np.where(live, (-rch + lh * rph) / sh, 0.0)
            tl = np.where(live, (-rcl + ll * rpl) / sl, 0.0)
            rhs = -rd - _rows_apply_T(T, th - tl)
            du = np.linalg.solve(Lc.T, np.linalg.solve(Lc, rhs))
            dz = _rows_apply(T, du)
            dsh = -rph - dz
            dsl = -rpl + dz
            dlh = np.where(live, (-rch - lh * dsh) / sh, 0.0)
            dll = np.where(live, (-rcl - ll * dsl) / sl, 0.0)
            return du, dsh, dsl, dlh, dll

        def max_step(v, dv):
            m = live & (dv < 0)
            return min(1.0, float((-v[m] / dv[m]).min())) if m.any() else 1.0

        du, dsh, dsl, dlh, dll = newton(lh * sh, ll * sl)
        a_aff = min(max_step(sh, dsh), max_step(sl, dsl), max_step(lh, dlh), max_step(ll, dll))
        mu_aff = float(((lh + a_aff * dlh) * (sh + a_aff * dsh) + (ll + a_aff * dll) * (sl + a_aff * dsl))[live].sum()) / nrow
        sigma = (mu_aff / mu) ** 3
        du, dsh, dsl, dlh, dll = newton(lh * sh + dsh * dlh - sigma * mu, ll * sl + dsl * dll - sigma * mu)
        def raw_step(v, dv):
            m = live & (dv < 0)
            return float((-v[m] / dv[m]).min()) if m.any() else np.inf

        frac = min(0.9999, max(0.99, 1.0 - 0.1 * (1.0 - a_aff) ** 2))   # fraction to the boundary, as in the kernel
        alpha = min(1.0, frac * min(raw_step(sh, dsh), raw_step(sl, dsl), raw_step(lh, dlh), raw_step(ll, dll)))
        u = u + alpha * du
        sh, sl = sh + alpha * dsh, sl + alpha * dsl
        lh, ll = lh + alpha * dlh, ll + alpha * dll
    # the cap: the kernel reports the last iterate it tested against the reduced tolerances as converged (the step
    # taken after that test is not undone, nor is the iterate it leads to tested)
    return result(max_iter, acceptable, "reduced" if acceptable else "cap")
