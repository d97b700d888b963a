"""Lagrangian particles without a device: the interpolation stencil, periodic wrap of unwrapped positions, the RK4
(Simpson) recurrence of an inertial oscillation, and the argument checks of the Python API."""
import types

import numpy as np
import pytest

import particles_ref as pr
from niwqg_b200 import _native as nat
from niwqg_b200.Particles import Particles


def test_weights_reproduce_cubics_exactly():
    rng = np.random.RandomState(0)
    a = rng.rand(1000)
    w = pr.weights(a)
    np.testing.assert_allclose(w.sum(-1), 1.0, rtol=0, atol=1e-15)
    nodes = np.arange(-1, 3, dtype=np.float64)
    for c in rng.randn(5, 4):
        p = lambda s: c[0] + c[1] * s + c[2] * s ** 2 + c[3] * s ** 3
        got = (w * p(nodes)).sum(-1)
        np.testing.assert_allclose(got, p(a), rtol=0, atol=1e-13 * np.abs(c).sum())
    # nodes: the weights are the unit vectors
    np.testing.assert_array_equal(pr.weights(0.0), [0.0, 1.0, 0.0, 0.0])


def test_interpolation_of_a_bicubic_field_is_exact_away_from_the_wrap():
    N, L = 32, 1.0e5
    dx = L / N
    xc = (np.arange(N) + 0.5) * dx
    X, Y = np.meshgrid(xc, xc)
    cx, cy = (0.3, -1.2, 0.7, 0.25), (1.1, 0.4, -0.6, 0.15)
    px = lambda x: sum(c * (x / L) ** k for k, c in enumerate(cx))
    py = lambda y: sum(c * (y / L) ** k for k, c in enumerate(cy))
    f = px(X) * py(Y)
    rng = np.random.RandomState(1)
    xy = (3 * dx + rng.rand(500, 2) * (L - 6 * dx))          # stencils stay inside the grid
    xy[:4] = [[3 * dx, 4 * dx], [10.5 * dx, 7 * dx], [20 * dx, 20.5 * dx], [28 * dx, 28 * dx]]   # edges, centres
    got = pr.interp(f, xy, L)
    np.testing.assert_allclose(got, px(xy[:, 0]) * py(xy[:, 1]), rtol=0, atol=1e-13)
    # complex fields: real and imaginary parts separately
    gc = pr.interp(f + 2j * f, xy, L)
    np.testing.assert_allclose(gc.imag, 2 * got, rtol=0, atol=1e-13)


def test_unwrapped_positions_interpolate_as_their_periodic_image():
    N, L = 64, 2 * np.pi * 2e5
    dx = L / N
    rng = np.random.RandomState(2)
    f = rng.randn(N, N)
    xy = rng.rand(300, 2) * L
    xy[:3] = [[0.0, 0.0], [0.5 * dx, L - 1e-9], [L - 0.5 * dx, dx]]
    for shift in (3 * L, -2 * L, 7 * L):
        i0, w0 = pr.stencil(xy[:, 0], L, N)
        i1, w1 = pr.stencil(xy[:, 0] + shift, L, N)
        # the same point up to the rounding of the shifted position: its fraction a moves by < 1e-12 (in cells)
        same = np.all(i0 == i1, axis=-1)
        assert same.mean() > 0.98
        np.testing.assert_allclose(w1[same], w0[same], rtol=0, atol=1e-12)
        a = pr.interp(f, xy, L)
        b = pr.interp(f, xy + shift, L)
        np.testing.assert_allclose(b, a, rtol=0, atol=1e-12 * np.abs(f).max() * 8)


def test_inertial_simpson_recurrence_matches_the_circle():
    f, dt, phi = 1.e-4, 2000.0, 0.07 - 0.05j
    R = abs(phi) / f
    n = 300
    z = pr.inertial_simpson(0.0, phi, f, dt, n)
    exact = pr.inertial_circle(0.0, phi, f, dt * np.arange(n + 1))
    err = np.abs(z - exact)
    bound = np.arange(n + 1) * (f * dt) ** 5 / 1440.0 * R
    assert np.all(err <= bound + 1e-12 * R)
    # clockwise for f > 0: the angle about the centre decreases
    c = exact[0] - 1j * phi / f
    ang = np.unwrap(np.angle(z - c))
    assert np.all(np.diff(ang) < 0)
    # the reference RK4 driver reduces to the same recurrence when the velocity only depends on time
    N, L = 16, 1e6
    stage = dict(u=np.zeros((N, N)), v=np.zeros((N, N)), phi=np.full((N, N), phi))
    xy = np.array([[0.3 * L, 0.6 * L]])
    t = 0.0
    for k in range(5):
        xy = pr.rk4_step(xy, [stage] * 4, L, 0.0, f, t, dt, True)
        t += dt
    zz = pr.inertial_simpson(complex(0.3 * L, 0.6 * L), phi, f, dt, 5)[-1]
    assert abs(complex(xy[0, 0], xy[0, 1]) - zz) < 1e-12 * R


class _FakeHandle(object):
    def __init__(self, model, nranks=1):
        self.nranks = nranks
        self.params = types.SimpleNamespace(model=model)
        self.calls = []

    def particles_set(self, xy, t, waves):
        self.calls.append((None if xy is None else xy.copy(), t, waves))

    def particles_count(self):
        return 0 if not self.calls or self.calls[-1][0] is None else self.calls[-1][0].shape[1]


class _FakeModel(Particles):
    def __init__(self, model=nat.MODEL_COUPLED, batch=1, nranks=1):
        self._h = _FakeHandle(model, nranks)
        self.batch, self.t = batch, 12.5


def test_positions_shapes_and_values_are_checked():
    a = nat.particle_positions([[1, 2], [3, 4]], 3)
    assert a.shape == (3, 2, 2) and a.dtype == np.float64 and a.flags.c_contiguous
    b = nat.particle_positions(np.zeros((3, 5, 2)), 3)
    assert b.shape == (3, 5, 2)
    for bad in (np.zeros((4,)), np.zeros((4, 3)), np.zeros((2, 5, 2)), np.zeros((3, 5, 2, 1)), np.zeros((0, 2)),
                [[1.0, np.nan]], [[np.inf, 0.0]], np.array([["a", "b"]]), np.zeros((3, 2), complex)):
        with pytest.raises(ValueError):
            nat.particle_positions(bad, 3)


def test_model_api_checks_before_the_device():
    m = _FakeModel(batch=2)
    m.set_particles([[1.0, 2.0]], waves=True)
    xy, t, waves = m._h.calls[-1]
    assert xy.shape == (2, 1, 2) and t == 12.5 and waves
    m.set_particles(None)
    assert m._h.calls[-1][0] is None
    with pytest.raises(ValueError):
        m.set_particles(np.zeros((3, 1, 2)))
    with pytest.raises(ValueError):
        m.set_particles([[0.0, np.nan]])
    with pytest.raises(ValueError):
        m.sample_particles("w")
    with pytest.raises(ValueError):
        m.sample_particles("q")               # no particles yet
    qg = _FakeModel(model=nat.MODEL_QG)
    with pytest.raises(ValueError):
        qg.set_particles([[0.0, 0.0]], waves=True)
    qg.set_particles([[0.0, 0.0]])
    with pytest.raises(ValueError):
        qg.sample_particles("phi")
    slab = _FakeModel(nranks=2)
    with pytest.raises(NotImplementedError):
        slab.set_particles([[0.0, 0.0]])
    with pytest.raises(NotImplementedError):
        slab.particles
    with pytest.raises(NotImplementedError):
        slab.sample_particles("q")
    assert slab._particles_state() is None
    assert m._h.calls[-1][0] is None          # the rejected calls reached nothing


def test_particle_abi_is_declared_and_exported():
    import os
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                            "niwqg_b200.h")).read()
    for n in ("niwqg_particles_set", "niwqg_particles_count", "niwqg_particles_get", "niwqg_particles_sample"):
        assert n in nat.EXPORTS and (n + "(") in hdr
