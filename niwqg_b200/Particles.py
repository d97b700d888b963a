"""Lagrangian particles (drifters) advected on the device with the model's own ETDRK4 stage velocities
(DESIGN.md section 3.4, niwqg_particles_* in include/niwqg_b200.h).

A particle is a point ``(x, y)`` in metres in the frame of the model's ``x, y`` (grid values at the cell centres
``(i + 1/2) dx``).  Positions are kept unwrapped, so displacements and pair separations can be read off directly;
interpolation reduces them modulo ``L``.  Every step moves the particles by classical RK4 whose four stages read the
fields of the model's own ETDRK4 stages, interpolated with the periodic 4-point (cubic) Lagrange stencil.  The
velocity is ``U + (u, v)``; with ``waves=True`` (models with a wave field) it also includes the near-inertial velocity
``u_w + i v_w = exp(-i f t) phi``, which draws the clockwise (f > 0) inertial loops of surface drifters.  In the Coupled
and QL models ``(u, v)`` is already the Lagrangian-mean flow, so ``waves=True`` counts the O(a^2) Stokes drift twice:
use ``waves=False`` for the mean transport, ``waves=True`` for drifter-like trajectories.

Particles change nothing on the model: fields, budgets and diagnostics are bit for bit those of a run without them.
Read the positions inside ``run_with_snapshots`` (``m.particles``) to record trajectories.
"""
import numpy as np

from . import _native as nat


class Particles(object):
    """Mixin of the model classes: ``set_particles``, ``particles``, ``sample_particles``."""

    _particles_waves = False

    def _particles_handle(self):
        if self._h.nranks > 1:
            raise NotImplementedError("particles on a slab-decomposed grid (nranks > 1): particles would have to "
                                      "migrate between ranks")
        return self._h

    def set_particles(self, xy, waves=False):
        """Seed particles at the positions ``xy`` (metres): shape ``(P, 2)`` seeds every member with the same P
        particles, ``(batch, P, 2)`` gives each member its own.  ``waves=True`` adds the wave velocity (not for
        QGModel).  ``set_particles(None)`` removes the particles.  The particle clock starts at the model's ``t``.
        ValueError for a wrong shape or a non-finite position."""
        h = self._particles_handle()
        if xy is None:
            h.particles_set(None, 0.0, False)
            self._particles_waves = False
            return
        if waves and self._h.params.model == nat.MODEL_QG:
            raise ValueError("waves=True needs a model with a wave field: QGModel has none")
        a = nat.particle_positions(xy, self.batch)
        h.particles_set(a, self.t, waves)
        self._particles_waves = bool(waves)

    def _particles_state(self):
        """(positions (batch, P, 2), clock, waves), or None without particles (checkpoints)."""
        if self._h.nranks > 1:
            return None
        xy, t = self._h.particles()
        return None if xy is None else (xy, t, self._particles_waves)

    def _set_particles_state(self, xy, t, waves):
        self._particles_handle().particles_set(nat.particle_positions(xy, self.batch), t, waves)
        self._particles_waves = bool(waves)

    @property
    def particles(self):
        """A copy of the current (unwrapped) positions: ``(P, 2)``, or ``(batch, P, 2)`` for an ensemble; None without
        particles."""
        xy, _ = self._particles_handle().particles()
        if xy is None:
            return None
        return xy[0] if self.batch == 1 else xy

    def sample_particles(self, name):
        """``name`` (q, u, v or phi) interpolated at the current positions with the particles' own stencil, from the
        array the attribute of that name returns: ``(P,)`` or ``(batch, P)``."""
        if name not in nat.PARTICLE_FIELDS:
            raise ValueError("sample_particles: name must be one of %s, got %r" % (sorted(nat.PARTICLE_FIELDS), name))
        h = self._particles_handle()
        if name == "phi" and self._h.params.model == nat.MODEL_QG:
            raise ValueError("sample_particles('phi'): QGModel has no wave field")
        if h.particles_count() == 0:
            raise ValueError("sample_particles: the model has no particles (set_particles first)")
        out = h.particles_sample(nat.PARTICLE_FIELDS[name])
        return out[0] if self.batch == 1 else out
