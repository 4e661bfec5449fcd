"""Nonlinear plant of the benchmark system: the cart-pole between two soft walls
(notebooks/cart_pole_with_walls/nonlinear_dynamics.py:1-118; SURVEY.md 8f-4), for closed loops against the true plant
instead of the linear MLD model + noise (statistical_analysis.py:176-194).

The reference derives the equations of motion symbolically (sympy Lagrangian) and lambdifies them; here they are written
out in closed form.  Coordinates q = (qc cart position, qp pole angle from the upright), pole tip at
(qc - l sin qp, l cos qp), point masses mc (cart) and mp (pole tip):

    [ mc + mp     -mp l cos qp ] [qc'']   [ fc + fl - fr - mp l sin(qp) qp'^2 ]
    [ -mp l cos qp     mp l^2  ] [qp''] = [ mp g l sin qp - l cos(qp) (fl - fr) ]

fl (fr) is the push of the left (right) wall on the pole tip, a spring-damper that acts only in penetration and only
when it pushes:  f = max(0, -stiffness * gap -/+ damping * tip velocity)  if gap <= 0.
"""
import numpy as np


def n_substeps(dt, h_des):
    """Euler sub-steps per sample of CartPoleWithWalls.simulate"""
    return max(1, int(round(dt / h_des)))


class CartPoleWithWalls(object):

    def __init__(self, mc=1., mp=1., l=1., d=.5, stiffness=100., damping=10., g=10.):
        self.mc, self.mp, self.l, self.d, self.k, self.c, self.g = mc, mp, l, d, stiffness, damping, g

    def params(self):
        """(mc, mp, l, d, stiffness, damping, g): the parameter set of the device plant (WSHMPC_PLANT_CARTPOLE_NPARAM)"""
        return np.array([self.mc, self.mp, self.l, self.d, self.k, self.c, self.g], dtype=float)

    def gaps(self, x):
        """distance of the pole tip from the left / right wall (negative in penetration)"""
        tip = x[..., 0] - self.l * np.sin(x[..., 1])
        return tip + self.d, self.d - tip

    def contact_forces(self, x):
        """(fl, fr) of nonlinear_dynamics.py:95-110"""
        gl, gr = self.gaps(x)
        vtip = x[..., 2] - self.l * np.cos(x[..., 1]) * x[..., 3]
        fl = -self.k * gl - self.c * vtip
        fr = -self.k * gr + self.c * vtip
        fl = np.where((gl > 0.) | (fl < 0.), 0., fl)
        fr = np.where((gr > 0.) | (fr < 0.), 0., fr)
        return fl, fr

    def x_dot(self, x, fc):
        """state derivative for x = (qc, qp, qc', qp') [..., 4] and cart force fc [...]"""
        mc, mp, l, g = self.mc, self.mp, self.l, self.g
        s, c = np.sin(x[..., 1]), np.cos(x[..., 1])
        fl, fr = self.contact_forces(x)
        r1 = fc + fl - fr - mp * l * s * x[..., 3] ** 2
        r2 = mp * g * l * s - l * c * (fl - fr)
        m11, m12, m22 = mc + mp, -mp * l * c, mp * l * l
        det = m11 * m22 - m12 * m12
        qcdd = (m22 * r1 - m12 * r2) / det
        qpdd = (m11 * r2 - m12 * r1) / det
        return np.stack((x[..., 2], x[..., 3], qcdd, qpdd), axis=-1)

    def simulate(self, x, dt, fc=0., h_des=.001):
        """explicit Euler with sub-steps of about h_des (nonlinear_dynamics.py:112-118); returns the state after dt.
        x [..., 4], fc [...] (held constant over dt)."""
        n = n_substeps(dt, h_des)
        h = dt / n
        x = np.array(x, dtype=float)
        fc = np.asarray(fc, dtype=float)
        for _ in range(n):
            x = x + h * self.x_dot(x, fc)
        return x

    def linearization(self):
        """(A_c, B_c) of x' = f(x, (fc, fl, fr)) at the upright equilibrium, B_c columns (fc, fl, fr)"""
        mc, mp, l, g = self.mc, self.mp, self.l, self.g
        Minv = np.linalg.inv(np.array([[mc + mp, -mp * l], [-mp * l, mp * l * l]]))
        A = np.zeros((4, 4)); A[0, 2] = A[1, 3] = 1.
        A[2:, 1] = Minv.dot([0., mp * g * l])
        B = np.zeros((4, 3))
        B[2:, 0] = Minv.dot([1., 0.]); B[2:, 1] = Minv.dot([1., -l]); B[2:, 2] = Minv.dot([-1., l])
        return A, B


class DevicePlant(object):
    """The cart-pole between soft walls integrated on the device (wshmpc_plant in include/wshmpc.h): what
    CartPoleWithWalls.simulate(x, dt, u[:, fc_index], h_des) computes, for a batch of states, in the closed loop
    (ClosedLoop(..., plant=DevicePlant(...))) or standalone (step).

    plants: one CartPoleWithWalls for every instance, or a list of them, one per instance (a robustness sweep over
    plant parameters).  The Euler sub-step count follows simulate: n_sub = max(1, round(dt / h_des))."""

    def __init__(self, plants, dt, h_des=1e-3, fc_index=0, device='cuda'):
        import torch
        ps = [plants] if isinstance(plants, CartPoleWithWalls) else list(plants)
        if not ps or not all(isinstance(p, CartPoleWithWalls) for p in ps):
            raise ValueError('plants: a CartPoleWithWalls or a non-empty list of them')
        if not dt > 0. or not h_des > 0.:
            raise ValueError('dt and h_des must be positive (dt = %r, h_des = %r)' % (dt, h_des))
        if int(fc_index) != fc_index or fc_index < 0:
            raise ValueError('fc_index must be a non-negative input index, got %r' % (fc_index,))
        self.dt, self.fc_index = float(dt), int(fc_index)
        self.n_sub = n_substeps(dt, h_des)
        self.params = torch.as_tensor(np.stack([p.params() for p in ps]), dtype=torch.float64, device=device).contiguous()

    @property
    def n_sets(self):
        return self.params.shape[0]

    def step(self, handle, x, u):
        """States after dt from x [n, 4] under inputs u [n, nu] (CUDA fp64 tensors); parameter set k for state k when
        there is one set per state (wshmpc_plant_step).  Asynchronous on the handle's stream."""
        return handle.plant_step(self, x, u)
