"""Host-side problem compiler: MLD system + controller data -> shared operator of the QP kernel.

north_star keeps "the MLD condensing" as host-side precomputation; this module is that step.  It is
run once per controller (numpy, fp64) and its output is uploaded once (csrc/wshmpc.cu wshmpc_create).

Math (DESIGN.md section "shared operator"): the node QP of controller.py:119-184 has variables
(x_t, u_t) tied by the dynamics rows.  Let xi = (z, X), z = (u_0..u_{T-1}), X = (x_1..x_T); the
dynamics rows confine xi to the affine subspace xi = P0 x0 + G z, G = [I; Gamma].  With the thin QR
G = N T the orthonormal coordinates y = T z give
    cost = 1/2 y'Hy y + (Fy x0)'y + const,     Hy = N' Hs N  (eigenvalues <= 2 max eig(Q'Q, R'R, Q_T'Q_T))
    rows : Ay y <= hbar - Ey x0  (mu rows, reference order) and  lb <= Sel N y <= ub  (nu_lb / nu_ub rows)
The kernel solves the proximal-regularised problem min 1/2 y'(Hy + eps I) y + ... in least-distance
form: with Rinv'(Hy + eps I) Rinv = I (symmetric eigen-decomposition, NOT Cholesky, so that the flat and
the curved directions are scaled column by column) and v = Rinv^-1 y + Rinv' f,
    min 1/2 |v|^2   s.t.   bl <= Mh v <= bu ,   Mh = rows of (Ay Rinv) normalised to unit length.
"""
import numpy as np


class RecordLayout(object):
    """Offsets (in doubles) of the per-node records, identical to wshmpc_layout (include/wshmpc.h):
    primal  x_0..x_T | u_0..u_{T-1} ;  dual  lam | mu | nu_lb | nu_ub | rho | sigma."""

    def __init__(self, T, nx, nu, nub, mc, nq, nqT, nr):
        self.primal = (T + 1) * nx + T * nu
        self.off_lam = 0
        self.off_mu = (T + 1) * nx
        self.off_nu_lb = self.off_mu + mc
        self.off_nu_ub = self.off_nu_lb + T * nub
        self.off_rho = self.off_nu_ub + T * nub
        self.off_sigma = self.off_rho + T * nq + nqT
        self.dual = self.off_sigma + T * nr
        # a tree's dual record: the duals, the proximal centre (T nu doubles), and one zero double if that sum is odd
        self.rec_stride = (self.dual + T * nu + 1) & ~1


class ProblemData(object):
    """All arrays the C ABI needs (contiguous fp64 / int32), plus sizes."""

    def __init__(self, A, B, F, G, h, nub, T, Q, R, Q_T, F_Tm1, G_Tm1, h_Tm1, M_mu, M_rho,
                 eps=None, tol_p=1e-7, tol_d=1e-12, tol_sing=1e-7, tol_ray=1e-9, prox_tol=1e-11,
                 max_iter=5000, max_prox=50):
        f = lambda M: np.ascontiguousarray(M, dtype=np.float64)
        self.A, self.B, self.F, self.G, self.h = f(A), f(B), f(F), f(G), f(h)
        self.Q, self.R, self.Q_T = f(Q), f(R), f(Q_T)
        self.F_Tm1, self.G_Tm1, self.h_Tm1 = f(F_Tm1), f(G_Tm1), f(h_Tm1)
        self.M_mu, self.M_rho = f(M_mu), f(M_rho)
        nx, nu = self.B.shape
        self.nx, self.nu, self.nub, self.nuc, self.T = nx, nu, int(nub), nu - int(nub), int(T)
        self.nh, self.nh1 = self.h.size, self.h_Tm1.size
        self.nq, self.nqT, self.nr = self.Q.shape[0], self.Q_T.shape[0], self.R.shape[0]
        self.n = self.T * nu
        self.nb = self.T * self.nub
        self.mc = (self.T - 1) * self.nh + self.nh1
        self.m = self.mc + self.nb
        self.tol_p, self.tol_d, self.tol_sing, self.tol_ray = tol_p, tol_d, tol_sing, tol_ray
        self.prox_tol, self.max_iter, self.max_prox = prox_tol, max_iter, max_prox
        self.layout = RecordLayout(self.T, nx, nu, self.nub, self.mc, self.nq, self.nqT, self.nr)
        self._build(eps)

    def _build(self, eps):
        T, nx, nu, nub, nuc, n = self.T, self.nx, self.nu, self.nub, self.nuc, self.n
        A, B = self.A, self.B
        # state maps X = Pbar x0 + Gbar z
        Gbar = np.zeros((T * nx, n)); Pbar = np.zeros((T * nx, nx))
        Pk = np.eye(nx); Gk = np.zeros((nx, n))
        for t in range(T):
            Gk = A.dot(Gk); Gk[:, t * nu:(t + 1) * nu] += B
            Pk = A.dot(Pk)
            Gbar[t * nx:(t + 1) * nx] = Gk; Pbar[t * nx:(t + 1) * nx] = Pk
        N, _ = np.linalg.qr(np.vstack((np.eye(n), Gbar)))
        ns = n + T * nx
        P0 = np.vstack((np.zeros((n, nx)), Pbar))
        # sparse-form Hessian and rows
        Hs = np.zeros((ns, ns))
        RtR, QtQ, QTtQT = self.R.T.dot(self.R), self.Q.T.dot(self.Q), self.Q_T.T.dot(self.Q_T)
        for t in range(T):
            Hs[t * nu:(t + 1) * nu, t * nu:(t + 1) * nu] = 2. * RtR
            o = n + t * nx
            Hs[o:o + nx, o:o + nx] = 2. * (QtQ if t < T - 1 else QTtQT)
        As = np.zeros((self.mc, ns)); E0 = np.zeros((self.mc, nx)); hbar = np.zeros(self.mc)
        r = 0
        for t in range(T):
            Ft, Gt, ht = (self.F, self.G, self.h) if t < T - 1 else (self.F_Tm1, self.G_Tm1, self.h_Tm1)
            k = ht.size
            As[r:r + k, t * nu:(t + 1) * nu] = Gt
            if t == 0:
                E0[r:r + k] = Ft
            else:
                As[r:r + k, n + (t - 1) * nx:n + t * nx] = Ft
            hbar[r:r + k] = ht
            r += k
        self.bin_idx = np.array([t * nu + nuc + i for t in range(T) for i in range(nub)], dtype=np.int32)
        Sel = np.zeros((self.nb, ns)); Sel[np.arange(self.nb), self.bin_idx] = 1.
        HsN = Hs.dot(N)
        Hy = N.T.dot(HsN); Hy = .5 * (Hy + Hy.T)
        Fy = HsN.T.dot(P0)
        Ay = np.vstack((As.dot(N), Sel.dot(N)))
        Ey = E0 + As.dot(P0)
        lamb, U = np.linalg.eigh(Hy)
        if eps is None:
            # 1% of the smallest non-zero curvature: the proximal outer loop contracts >= 100x / iteration
            pos = lamb[lamb > 1e-9 * lamb.max()]
            eps = 1e-2 * float(pos.min())
        self.eps = float(eps)
        Rinv = U / np.sqrt(np.maximum(lamb, 0.) + self.eps)[None, :]
        # Rinv is fixed only up to an orthogonal factor on the right.  Choose it so that the bound rows of
        # the binaries, taken in chronological order (t, i) -- the order branch_in_time pins them in,
        # controller.py:13-44 -- are LOWER TRIANGULAR in v: row j has its non-zeros in columns 0..j.  A node
        # whose first d binaries are pinned then fixes v[:d] by one forward substitution and the kernel
        # solves its QP in the remaining n - d coordinates (working set, factor and pricing all shrink).
        M = Ay.dot(Rinv)
        nrm = np.linalg.norm(M, axis=1); nrm[nrm == 0.] = 1.
        nb = self.nb
        Qrot, Rr = np.linalg.qr((M[self.mc:] / nrm[self.mc:, None]).T, mode='complete')
        sgn = np.sign(np.diag(Rr[:nb, :nb])); sgn[sgn == 0.] = 1.
        Qrot[:, :nb] *= sgn[None, :]
        Rinv = Rinv.dot(Qrot)
        M = Ay.dot(Rinv)
        for j in range(nb):
            M[self.mc + j, j + 1:] = 0.
        nrm = np.linalg.norm(M, axis=1); nrm[nrm == 0.] = 1.
        L = M[self.mc:, :nb] / nrm[self.mc:, None]
        dg = np.abs(np.diag(L))
        bad = np.nonzero(dg < 1e-6)[0]
        self.n_elim = int(bad[0]) if bad.size else nb
        Linv = np.zeros((nb, nb))
        if self.n_elim:
            Linv[:self.n_elim, :self.n_elim] = np.tril(np.linalg.inv(L[:self.n_elim, :self.n_elim]))
        self.Linv = np.ascontiguousarray(Linv)
        arow = np.concatenate((np.linalg.norm(As, axis=1), np.ones(self.nb)))
        c = np.ascontiguousarray
        self.Mh = c(M / nrm[:, None]); self.nrm = c(nrm); self.vscale = c(nrm / np.maximum(1., arow))
        self.Eh = c(Ey / nrm[:self.mc, None]); self.hh = c(hbar / nrm[:self.mc])
        self.Rinv = c(Rinv); self.Kx = c(Rinv.T.dot(Fy)); self.Zmap = c(N[:n])
        self.Wf = c(N.dot(Rinv)); self.ns = ns

    @staticmethod
    def from_controller_data(mld, T, objective, F_Tm1, G_Tm1, h_Tm1, M_mu, M_rho, **kw):
        Q, R, Q_T = objective
        return ProblemData(mld.A, mld.B, mld.F, mld.G, mld.h, mld.nub, T, Q, R, Q_T,
                           F_Tm1, G_Tm1, h_Tm1, M_mu, M_rho, **kw)
