"""TEST-ONLY reference for the constraint solve: MuJoCo's soft-constraint problem solved in its dual form by a generic convex method,
sharing no formula with the primal Newton solvers (engine.cuh solve / newton_iteration, ur3e_oracle.c solve_newton).

At a state the constraint rows (J, R, aref, types, friction-loss bounds, the contacts' friction) are input; the forces are the
unique minimiser of

    D(f) = 1/2 f^T (A + R) f + f^T (J qacc_smooth - aref),   A = J M^-1 J^T,   f in Omega

with Omega the product of one set per row group: equality rows free, friction-loss rows |f| <= frictionloss, limit rows f >= 0, and
each elliptic contact the cone f_n >= |(f_1 / mu_1, f_2 / mu_2)| (mu_1, mu_2 = the pair's friction[0:2]).  The accelerations are
qacc = qacc_smooth + M^-1 J^T f.

The solve runs in the scaled variables g = R^1/2 f, where the problem is min 1/2 g^T (S A S + I) g + g^T S (J qacc_smooth - aref),
S = R^-1/2.  There the contact cone is circular: |g_t| <= mu g_n with mu = mu_1 sqrt(R_1 / R_n), because the friction rows' R
satisfy R_1 mu_1^2 = R_2 mu_2^2 (checked per contact); friction loss is the box |g| <= F sqrt(R) and a limit g >= 0.  Each set has a
closed-form Euclidean projection, and the method is accelerated projected gradient with the exact strong-convexity momentum
(the Hessian's extreme eigenvalues are computed) and gradient restarts, to 1e-9, then a semismooth Newton polish of the fixed-point
equation g = Pi(g - grad) (the projection's generalised Jacobian), kept only where it lowers the fixed-point residual.  The answer is
accepted only with a KKT certificate in the unscaled variables: f in Omega, y = (A + R) f + J qacc_smooth - aref in the dual set
(y = 0 on equality rows, the sign conditions of the friction-loss box, y >= 0 on limits, y_n >= |(mu_1 y_1, mu_2 y_2)| on contacts)
and f^T y = 0 per group, every residual relative to the problem's scale.

primal_cost(qacc) evaluates the primal objective through the per-group conjugates of the same sets,
s_b(x) = max_{f in Omega_b} (-f^T x - 1/2 f^T R f) = Pi(w)^T w - 1/2 |Pi(w)|^2 with w = -S x and Pi the scaled projection, so that
the duality gap P(qacc) + D(f*) grades any build's qacc without trusting either solver.
"""
import numpy as np

EQUALITY, FRICTION, LIMIT, CONTACT = 0, 1, 3, 7


class Problem:
    """One constraint problem.  cones: [(row address, mu_1, mu_2)] of the contacts (three rows each: normal, two tangents)."""

    def __init__(self, M, J, R, aref, qacc_smooth, types, frictionloss, cones):
        self.M = np.asarray(M, dtype=np.float64); self.J = np.asarray(J, dtype=np.float64).reshape(-1, self.M.shape[0])
        self.R = np.asarray(R, dtype=np.float64); self.aref = np.asarray(aref, dtype=np.float64)
        self.a0 = np.asarray(qacc_smooth, dtype=np.float64); self.types = np.asarray(types, dtype=np.int64)
        self.floss = np.asarray(frictionloss, dtype=np.float64); self.cones = [(int(a), float(m1), float(m2)) for a, m1, m2 in cones]
        n = len(self.R)
        assert self.J.shape[0] == n == len(self.aref) == len(self.types) == len(self.floss)
        assert np.all(self.R > 0)
        self.eq = np.flatnonzero(self.types == EQUALITY); self.fl = np.flatnonzero(self.types == FRICTION)
        self.lim = np.flatnonzero(self.types == LIMIT)
        self.cn = np.array([a for a, _, _ in self.cones], dtype=np.int64)
        self.mu12 = np.array([[m1, m2] for _, m1, m2 in self.cones]).reshape(-1, 2)
        covered = np.concatenate([self.eq, self.fl, self.lim, self.cn, self.cn + 1, self.cn + 2])
        assert np.array_equal(np.sort(covered), np.arange(n)), "every row belongs to exactly one group"
        assert np.all(self.types[self.cn] == CONTACT) and np.all(self.types[self.cn + 1] == CONTACT) and np.all(self.types[self.cn + 2] == CONTACT)
        # the circular cone of the scaled variables: |g_t| <= mu g_n
        Rn, R1, R2 = self.R[self.cn], self.R[self.cn + 1], self.R[self.cn + 2]
        self.mu = self.mu12[:, 0] * np.sqrt(R1 / Rn) if len(self.cn) else np.zeros(0)
        if len(self.cn):
            mu2 = self.mu12[:, 1] * np.sqrt(R2 / Rn)
            assert np.allclose(mu2, self.mu, rtol=1e-12, atol=0), "R_1 mu_1^2 != R_2 mu_2^2: the scaled cone is not circular"
        self.s = 1.0 / np.sqrt(self.R)
        L = np.linalg.cholesky(self.M)
        self.MinvJt = np.linalg.solve(L.T, np.linalg.solve(L, self.J.T))                  # M^-1 J^T
        self.A = self.J @ self.MinvJt
        self.A = 0.5 * (self.A + self.A.T)
        self.b = self.J @ self.a0 - self.aref                                             # J qacc_smooth - aref

    # ---------------------------------------------------------------------------------------------- scaled sets
    def project(self, g):
        """Euclidean projection of g [nefc] onto the scaled set K."""
        p = g.copy()
        if len(self.fl):
            bound = self.floss[self.fl] * np.sqrt(self.R[self.fl])
            p[self.fl] = np.clip(g[self.fl], -bound, bound)
        if len(self.lim):
            p[self.lim] = np.maximum(g[self.lim], 0.0)
        if len(self.cn):
            n = g[self.cn]; t = np.stack([g[self.cn + 1], g[self.cn + 2]], 1); tn = np.linalg.norm(t, axis=1); mu = self.mu
            a = (n + mu * tn) / (1.0 + mu * mu)
            inside = tn <= mu * n
            polar = mu * tn <= -n
            with np.errstate(invalid="ignore", divide="ignore"):
                scale = np.where(tn > 0, mu * a / np.where(tn > 0, tn, 1.0), 0.0)
            pn = np.where(inside, n, np.where(polar, 0.0, a))
            pt = np.where(inside[:, None], t, np.where(polar[:, None], 0.0, t * scale[:, None]))
            p[self.cn] = pn; p[self.cn + 1] = pt[:, 0]; p[self.cn + 2] = pt[:, 1]
        return p

    # ---------------------------------------------------------------------------------------------- objective pieces
    def dual_cost(self, f):
        return 0.5 * f @ ((self.A + np.diag(self.R)) @ f) + f @ self.b

    def qacc(self, f):
        return self.a0 + self.MinvJt @ f

    def primal_cost(self, qacc):
        """P(qacc) = 1/2 (qacc - a0)^T M (qacc - a0) + sum_b s_b(J qacc - aref), s_b the conjugate of the group's set (see above)."""
        dq = np.asarray(qacc, dtype=np.float64) - self.a0
        w = -self.s * (self.J @ np.asarray(qacc, dtype=np.float64) - self.aref)
        p = self.project(w)
        return 0.5 * dq @ (self.M @ dq) + p @ w - 0.5 * p @ p

    # ---------------------------------------------------------------------------------------------- the solve
    def solve(self, tol=1e-9, max_iter=200000):
        n = len(self.R)
        if n == 0:
            self.f = np.zeros(0); return self.f
        H = self.s[:, None] * self.A * self.s[None, :] + np.eye(n)
        c = self.s * self.b
        ev = np.linalg.eigvalsh(H)
        Lc, mc = ev[-1], ev[0]
        q = np.sqrt(mc / Lc)
        beta = (1.0 - q) / (1.0 + q)
        scale = max(np.abs(c).max(), 1e-300)
        g = self.project(-c / Lc); y = g.copy()
        for it in range(max_iter):
            gn = self.project(y - (H @ y + c) / Lc)
            if it % 16 == 0:
                r = np.abs(gn - self.project(gn - (H @ gn + c) / Lc)).max() * Lc
                if r <= tol * scale:
                    g = gn
                    break
            # adaptive restart (gradient scheme): drop the momentum when it points uphill
            if (H @ y + c) @ (gn - g) > 0:
                y = gn.copy()
            else:
                y = gn + beta * (gn - g)
            g = gn
        self.iters = it
        g = self._polish(H, c, g)
        self.g = g
        self.f = self.s * g
        return self.f

    def _polish(self, H, c, g):
        """Semismooth Newton on F(g) = g - Pi(g - (H g + c)) from the first-order point: the projection's generalised Jacobian
        fixes the rows on a bound, leaves interior rows free and moves cone-boundary contacts along the boundary.  The best
        iterate by fixed-point residual is kept."""
        def resid(x):
            return np.abs(x - self.project(x - (H @ x + c))).max()
        best, rb = g, resid(g)
        x = g
        for _ in range(20):
            z = x - (H @ x + c)
            P = self._proj_jacobian(z)
            # fixed point x = Pi(z(x)): Newton on F(x) = x - Pi(x - Hx - c), dF = I - P (I - H)
            F = x - self.project(z)
            dF = np.eye(len(x)) - P @ (np.eye(len(x)) - H)
            try:
                dx = np.linalg.solve(dF, -F)
            except np.linalg.LinAlgError:
                break
            x = x + dx
            r = resid(x)
            if r < rb:
                best, rb = x.copy(), r
            if r == 0.0:
                break
        return self.project(best)

    def _proj_jacobian(self, z):
        n = len(z); P = np.eye(n)
        if len(self.fl):
            bound = self.floss[self.fl] * np.sqrt(self.R[self.fl])
            P[self.fl, self.fl] = (np.abs(z[self.fl]) < bound).astype(float)
        if len(self.lim):
            P[self.lim, self.lim] = (z[self.lim] > 0).astype(float)
        for k, a in enumerate(self.cn):
            nn, t = z[a], z[a + 1:a + 3]; tn = np.linalg.norm(t); mu = self.mu[k]
            idx = [a, a + 1, a + 2]
            if tn <= mu * nn:
                continue
            if mu * tn <= -nn or tn == 0.0:
                P[np.ix_(idx, idx)] = 0.0
                continue
            u = t / tn; al = (nn + mu * tn) / (1 + mu * mu)
            J = np.zeros((3, 3))
            J[0, 0] = 1 / (1 + mu * mu); J[0, 1:] = mu * u / (1 + mu * mu)
            J[1:, 0] = mu * u / (1 + mu * mu)
            J[1:, 1:] = mu * mu * np.outer(u, u) / (1 + mu * mu) + mu * al / tn * (np.eye(2) - np.outer(u, u))
            P[np.ix_(idx, idx)] = J
        return P

    # ---------------------------------------------------------------------------------------------- certificate and census
    def certificate(self, f=None):
        """{group: worst relative residual} of the KKT conditions at f (default: the solution), in the unscaled variables."""
        f = self.f if f is None else f
        y = (self.A + np.diag(self.R)) @ f + self.b
        fs = max(np.abs(f).max(initial=0.0), 1e-300)
        ys = max(np.abs(self.A @ f).max(initial=0.0), np.abs(self.R * f).max(initial=0.0), np.abs(self.b).max(initial=0.0), 1e-300)
        out = dict(equality=0.0, friction=0.0, limit=0.0, contact=0.0)
        if len(self.eq):
            out["equality"] = np.abs(y[self.eq]).max() / ys
        for i in self.fl:
            F = self.floss[i]
            feas = max(abs(f[i]) - F, 0.0) / fs
            free = abs(y[i]) / ys                                                          # |f| < F: y = 0
            bound = (F - abs(f[i])) / fs + max(np.sign(f[i]) * y[i], 0.0) / ys             # f = +-F: y of the opposite sign
            out["friction"] = max(out["friction"], feas + min(free, bound))
        for i in self.lim:
            out["limit"] = max(out["limit"], max(-f[i], 0.0) / fs, max(-y[i], 0.0) / ys, min(f[i] / fs, y[i] / ys))
        for k, a in enumerate(self.cn):
            m1, m2 = self.mu12[k]
            feas = max(np.hypot(f[a + 1] / m1, f[a + 2] / m2) - f[a], 0.0) / fs
            dual = max(np.hypot(m1 * y[a + 1], m2 * y[a + 2]) - y[a], 0.0) / ys
            comp = abs(f[a:a + 3] @ y[a:a + 3]) / (fs * ys)
            out["contact"] = max(out["contact"], feas, dual, comp)
        return out

    def census(self, rel=1e-9):
        """Zones of the optimum: contacts sticking (strictly inside the cone), sliding (on the cone, f_n > 0) or separated (f = 0);
        friction-loss rows saturated or linear; limits active or inactive."""
        f = self.f
        fs = max(np.abs(f).max(initial=0.0), 1e-300)
        c = dict(sticking=0, sliding=0, separated=0, friction_saturated=0, friction_linear=0, limit_active=0, limit_inactive=0,
                 equality=len(self.eq))
        for k, a in enumerate(self.cn):
            m1, m2 = self.mu12[k]
            if f[a] <= rel * fs:
                c["separated"] += 1
            elif np.hypot(f[a + 1] / m1, f[a + 2] / m2) < f[a] * (1 - 1e-6):
                c["sticking"] += 1
            else:
                c["sliding"] += 1
        for i in self.fl:
            c["friction_saturated" if abs(f[i]) >= self.floss[i] * (1 - 1e-9) else "friction_linear"] += 1
        for i in self.lim:
            c["limit_active" if f[i] > rel * fs else "limit_inactive"] += 1
        return c

    def contact_forces(self, f=None):
        f = self.f if f is None else f
        return np.array([f[a:a + 3] for a in self.cn]).reshape(-1, 3)


def from_oracle(d):
    """The problem at the oracle's state after d.forward(): rows, mass matrix and qacc_smooth only (never its qacc or forces)."""
    nv, nefc = d.m.nv, d.nefc
    cones = [(c.efc_address, c.friction[0], c.friction[1]) for c in d.contacts() if c.efc_address >= 0]
    for c in d.contacts():
        assert c.efc_address < 0 or c.dim == 3
    return Problem(d.fullM(), np.asarray(d.efc_J)[:nefc * nv], np.asarray(d.efc_R)[:nefc], np.asarray(d.efc_aref)[:nefc],
                   np.asarray(d.qacc_smooth), np.asarray(d.efc_type)[:nefc], np.asarray(d.efc_frictionloss)[:nefc], cones)


_CACHE = {}


def reference(xml, qpos, qvel, ctrl):
    """(oracle Data after forward(), solved Problem) at a state; cached per state within the process.  The warm start plays no part
    in the problem, so it is not an input."""
    from oracle import oracle as O
    key = (xml, np.asarray(qpos, dtype=np.float64).tobytes(), np.asarray(qvel, dtype=np.float64).tobytes(), np.asarray(ctrl, dtype=np.float64).tobytes())
    if key not in _CACHE:
        if ("model", xml) not in _CACHE:
            _CACHE[("model", xml)] = O.Model(xml)
        m = _CACHE[("model", xml)]
        d = O.Data(m); d.reset(); d.set_state(qpos, qvel); d.ctrl[:] = ctrl; d.forward()
        p = from_oracle(d)
        p.solve()
        _CACHE[key] = (d, p)
    return _CACHE[key]
