"""Numpy reference of the Lagrangian particles (niwqg_b200/csrc/kernels_particles.cuh, DESIGN.md section 3.4).

- ``weights`` / ``interp``: the periodic tensor-product 4-point (cubic) Lagrange interpolation, rows summed with the x
  weights and then the rows with the y weights, both in index order, as the kernel does.
- ``StageRecorder``: oracle subclasses that record the fields a particle sees at each ETDRK4 stage (u, v and phi when
  ``jacobian_psi_q`` runs at the start of a stage; YBJ, whose u, v are frozen and whose phi stays stale through the
  stages, records at ``_grad_phi``, its first call of a stage).  The pinned oracle is not changed.
- ``rk4_step`` / ``drive``: classical RK4 on the positions with those stage fields.
"""
import numpy as np

from oracle import niwqg_oracle as orc


def weights(a):
    """The 4 weights of nodes i-1 .. i+2 at the fraction a in [0, 1) (array or scalar): shape a.shape + (4,)."""
    a = np.asarray(a, np.float64)
    return np.stack([-a * (a - 1.0) * (a - 2.0) / 6.0,
                     (a + 1.0) * (a - 1.0) * (a - 2.0) / 2.0,
                     -(a + 1.0) * a * (a - 2.0) / 2.0,
                     (a + 1.0) * a * (a - 1.0) / 6.0], axis=-1)


def stencil(x, L, N):
    """Wrapped node indices (..., 4) and weights (..., 4) of the coordinate x (metres, unwrapped)."""
    x = np.asarray(x, np.float64)
    dx = L / N
    xr = x - np.floor(x / L) * L
    s = xr / dx - 0.5
    i = np.floor(s)
    a = s - i
    idx = (i.astype(np.int64)[..., None] + np.arange(-1, 3)) % N
    return idx, weights(a)


def interp(f, xy, L):
    """f: (N, N) array [iy][ix] (real or complex); xy: (..., 2) positions -> f at xy, shape xy.shape[:-1]."""
    N = f.shape[0]
    ix, wx = stencil(xy[..., 0], L, N)
    iy, wy = stencil(xy[..., 1], L, N)
    rows = []
    for j in range(4):
        g = f[iy[..., j][..., None], ix]                       # (..., 4) columns of row j
        r = wx[..., 0] * g[..., 0] + wx[..., 1] * g[..., 1] + wx[..., 2] * g[..., 2] + wx[..., 3] * g[..., 3]
        rows.append(r)
    return wy[..., 0] * rows[0] + wy[..., 1] * rows[1] + wy[..., 2] * rows[2] + wy[..., 3] * rows[3]


def velocity(stage, xy, L, U, f, t, waves):
    """(P, 2) velocity U + (u, v) [+ Re/Im exp(-i f t) phi] of one stage's fields {u, v, phi} at xy."""
    uvi = interp(stage["u"] + 1j * stage["v"], xy, L)
    vx, vy = U + uvi.real, uvi.imag
    if waves:
        ph = interp(stage["phi"], xy, L)
        cs, sn = np.cos(f * t), np.sin(f * t)
        vx = vx + (cs * ph.real + sn * ph.imag)
        vy = vy + (cs * ph.imag - sn * ph.real)
    return np.stack([vx, vy], axis=-1)


def rk4_step(xy, stages, L, U, f, t, dt, waves):
    """One RK4 step from the 4 stage fields (times t, t + dt/2, t + dt/2, t + dt)."""
    k1 = velocity(stages[0], xy, L, U, f, t, waves)
    k2 = velocity(stages[1], xy + 0.5 * dt * k1, L, U, f, t + 0.5 * dt, waves)
    k3 = velocity(stages[2], xy + 0.5 * dt * k2, L, U, f, t + 0.5 * dt, waves)
    k4 = velocity(stages[3], xy + dt * k3, L, U, f, t + dt, waves)
    return xy + (dt / 6.0) * (k1 + 2.0 * k2 + 2.0 * k3 + k4)


class _Record(object):
    def _record(self):
        phi = getattr(self, "phi", None)
        self.stages.append(dict(u=np.array(self.u, np.float64), v=np.array(self.v, np.float64),
                                phi=None if phi is None else np.array(phi)))


class NIWRecorder(_Record, orc.NIWQGOracle):
    """NIWQGOracle that records the stage fields of every step in ``self.stages``."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.stages = []

    def jacobian_psi_q(self):
        out = super().jacobian_psi_q()      # sets u, v of this stage; phi is this stage's
        self._record()
        return out

    def _grad_phi(self):                    # YBJ only: first call of each stage (frozen u, v; stale phi)
        super()._grad_phi()
        self._record()


class QGRecorder(_Record, orc.QGOracle):
    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.stages = []

    def jacobian_psi_q(self):
        out = super().jacobian_psi_q()
        self._record()
        return out


def drive(o, xy, nsteps, waves=False, step=None):
    """Step the recording oracle ``o`` nsteps times (``step``: its step function, default step_forward) and move the
    particles xy (P, 2) along.  Returns the positions after every step, (nsteps, P, 2)."""
    step = step or o.step_forward
    f = getattr(o, "f", 0.0)
    out = []
    t = float(o.t)
    for _ in range(nsteps):
        o.stages = []
        step()
        assert len(o.stages) == 4, len(o.stages)
        xy = rk4_step(xy, o.stages, o.L, o.U, f, t, o.dt, waves)
        t += o.dt
        out.append(xy)
    return np.array(out)


def inertial_simpson(z0, phi, f, dt, nsteps, t0=0.0):
    """The RK4 recurrence for a velocity exp(-i f t) phi that depends on time only (Simpson's rule): complex
    positions z_n = x_n + i y_n, n = 0 .. nsteps."""
    z = [complex(z0)]
    t = t0
    for _ in range(nsteps):
        w0, wh, w1 = (np.exp(-1j * f * s) * phi for s in (t, t + 0.5 * dt, t + dt))
        z.append(z[-1] + dt / 6.0 * (w0 + 4.0 * wh + w1))
        t += dt
    return np.array(z)


def inertial_circle(z0, phi, f, t, t0=0.0):
    """Exact trajectory of dz/dt = exp(-i f t) phi: a clockwise circle (f > 0) of radius |phi| / f."""
    t = np.asarray(t, np.float64)
    return z0 + 1j * phi / f * (np.exp(-1j * f * t) - np.exp(-1j * f * t0))
