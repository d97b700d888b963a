"""Stand-alone barotropic QG model (niwqg/QGModel.py) on the CUDA backend: rfft2-layout
spectral state, optional passive scalar, same constructor / set_q / set_c / run API."""
import logging

import numpy as np
from numpy import pi

from . import _native as nat
from . import Checkpoint
from .Particles import Particles
from .Kernel import _DeviceField, _Scalar, _LazyGrid, _wv2i
from .Diagnostics import add_diagnostic, increment_diagnostics
from .Saving import initialize_save_snapshots, save_setup, save_snapshots, save_diagnostics


class Model(Particles):
    """Parameters: niwqg/QGModel.py:65-91, plus ``batch`` and ``device``.  With batch > 1, each of U, beta, nu, nu4,
    mu, nu4c, nuc, muc may be a sequence of batch values, one per member; nx, L, dt, use_filter, dealias and
    passive_scalar are common to all members."""

    q = _DeviceField("Q"); qh = _DeviceField("QH"); p = _DeviceField("P"); ph = _DeviceField("PH")
    u = _DeviceField("U"); v = _DeviceField("V")
    filtr = _DeviceField("FILTR")
    expch = _DeviceField("EXPCH"); expch_h = _DeviceField("EXPCH_H"); Qh = _DeviceField("QHCOEF")
    f0 = _DeviceField("F0"); fab = _DeviceField("FAB"); fc = _DeviceField("FC")
    Ke = _Scalar("KE")
    _checkpoint_params = ("L", "dt", "U", "nu4", "nu", "mu", "beta", "passive_scalar", "nu4c", "nuc", "muc",
                          "use_filter", "dealias")
    _checkpoint_run = ("twrite", "tswrite", "tmax", "tdiags", "tsave_snapshots", "save_to_disk", "overwrite", "path")
    _checkpoint_attr = {"tsave_snapshots": "tsnaps"}

    def __init__(self, nx=128, ny=None, L=5e5, dt=10000., twrite=1000, tswrite=10, tmax=250000., use_filter=True,
                 U=.0, nu4=5.e9, nu=0, mu=0, beta=0, passive_scalar=False, nu4c=5.e9, nuc=0, muc=0, dealias=False,
                 save_to_disk=False, overwrite=True, tsave_snapshots=10, tdiags=10, path='output/', use_mkl=False,
                 nthreads=1, batch=1, device=0):
        kw = nat.member_keywords(batch, dict(U=U, beta=beta, nu=nu, nu4=nu4, mu=mu, nu4c=nu4c, nuc=nuc, muc=muc),
                                 dict(nx=nx, L=L, dt=dt, use_filter=use_filter, dealias=dealias,
                                      passive_scalar=passive_scalar))
        U, beta, nu, nu4, mu, nu4c, nuc, muc = (kw[k] for k in ("U", "beta", "nu", "nu4", "mu", "nu4c", "nuc", "muc"))
        self.nx = nx
        self.ny = nx
        self.L = L
        self.W = L
        self.dt = dt
        self.twrite = twrite
        self.tswrite = tswrite
        self.tmax = tmax
        self.tdiags = tdiags
        self.passive_scalar = passive_scalar
        self.dealias = dealias
        self.U, self.beta, self.nu4, self.nu, self.mu = U, beta, nu4, nu, mu
        self.nu4c, self.nuc, self.muc = nu4c, nuc, muc
        self.save_to_disk = save_to_disk
        self.overwrite = overwrite
        self.tsnaps = tsave_snapshots
        self.path = path
        self.use_filter = use_filter
        self.use_mkl = use_mkl
        self.nthreads = nthreads
        self.batch = batch
        self.device = device

        self._initialize_logger()
        self._initialize_grid()
        self._h = nat.Handle(model=nat.MODEL_QG, nx=nx, batch=batch, device=device, L=L, dt=dt, U=U, f=0.0, N=1.0,
                             m=0.0, nu=nu, nu4=nu4, mu=mu, nuw=0.0, nu4w=0.0, muw=0.0, beta=beta,
                             use_filter=int(bool(use_filter)), dealias=int(bool(dealias)),
                             passive_scalar=int(bool(passive_scalar)), nu4c=nu4c, nuc=nuc, muc=muc)
        self.t = 0
        self.tc = 0
        initialize_save_snapshots(self, self.path)
        save_setup(self, )
        self.cflmax = .5                          # niwqg/QGModel.py:135
        self.fft = lambda x: self._h.fft2(x, nat.FFT_R2C)     # niwqg/QGModel.py:551-552
        self.ifft = lambda x: self._h.fft2(x, nat.FFT_C2R)
        self._initialize_diagnostics()

    @property
    def c(self):
        return self._h.field("C") if self.passive_scalar else 0.

    @property
    def ch(self):
        return self._h.field("CH") if self.passive_scalar else 0.

    @property
    def cvar(self):
        if not self.passive_scalar:
            return 0.
        v = self._h.scalars()[:, nat.S["CVAR"]]
        return float(v[0]) if self.batch == 1 else v

    # whole-grid host arrays of niwqg/QGModel.py:232-269, built on first use (the device recomputes wavenumbers itself)
    x = _LazyGrid("x", lambda s: np.meshgrid(np.arange(0.5, s.nx, 1.) / s.nx * s.L, np.arange(0.5, s.ny, 1.) / s.ny * s.W)[0])
    y = _LazyGrid("y", lambda s: np.meshgrid(np.arange(0.5, s.nx, 1.) / s.nx * s.L, np.arange(0.5, s.ny, 1.) / s.ny * s.W)[1])
    k = _LazyGrid("k", lambda s: np.meshgrid(s.kk, s.ll)[0])
    l = _LazyGrid("l", lambda s: np.meshgrid(s.kk, s.ll)[1])
    ik = _LazyGrid("ik", lambda s: 1j * s.k)
    il = _LazyGrid("il", lambda s: 1j * s.l)
    wv2 = _LazyGrid("wv2", lambda s: s.k ** 2 + s.l ** 2)
    wv = _LazyGrid("wv", lambda s: np.sqrt(s.wv2))
    wv4 = _LazyGrid("wv4", lambda s: s.wv2 ** 2)
    wv2i = _LazyGrid("wv2i", _wv2i)

    def _initialize_grid(self):
        """Scalars and 1-D arrays of niwqg/QGModel.py:232-269 (half spectrum: nk = nx/2 + 1)."""
        self.dk = 2. * pi / self.L
        self.dl = 2. * pi / self.L
        self.nl = self.ny
        self.nk = self.nx // 2 + 1
        self.ll = self.dl * np.append(np.arange(0., self.nx / 2), np.arange(-self.nx / 2, 0.))
        self.kk = self.dk * np.arange(0., self.nk)
        self.dx = self.L / self.nx
        self.dy = self.W / self.ny
        self.M = self.nx * self.ny

    def _initialize_logger(self):
        self.logger = logging.getLogger(__name__)
        fhandler = logging.StreamHandler()
        fhandler.setFormatter(logging.Formatter('%(levelname)s: %(message)s'))
        if not self.logger.handlers:
            self.logger.addHandler(fhandler)
        self.logger.setLevel(10)
        self.logger.propagate = False
        self.logger.info(' Logger initialized')

    # ------------------------------------------------------------------ driver
    def run_with_snapshots(self, tsnapstart=0., tsnapint=432000.):
        tsnapints = np.ceil(tsnapint / self.dt)
        while (self.t < self.tmax):
            self._step_forward()
            if self.t >= tsnapstart and (self.tc % tsnapints) == 0:
                yield self.t
        return

    def _snapshot_fields(self):
        return ['t', 'q', 'c'] if self.passive_scalar else ['t', 'q']

    def run(self):
        """niwqg/QGModel.py:180-203."""
        if self.save_to_disk:
            save_snapshots(self, fields=self._snapshot_fields())
        while (self.t < self.tmax):
            self._step_forward()
        if self.save_to_disk:
            save_diagnostics(self)

    def _step_forward(self):
        """niwqg/QGModel.py:205-217."""
        self._step_etdrk4()
        increment_diagnostics(self, )
        self._print_status()
        save_snapshots(self, fields=self._snapshot_fields())

    def _step_etdrk4(self):
        """niwqg/QGModel.py:328-407 on the device."""
        self._h.step(1)

    def step(self, nsteps=1):
        self._h.step(nsteps)
        for _ in range(int(nsteps)):
            self.tc += 1
            self.t += self.dt

    def set_q(self, q=None):
        """niwqg/QGModel.py:507-520.  ``q=None`` (extension): the array queued with ``stage_inputs``."""
        self._h.set_q(q)

    def stage_inputs(self, q=None):
        """Extension: start the upload of the next ``set_q()`` argument now (see Kernel.stage_inputs)."""
        if q is not None:
            self._h.stage_q(q)

    def set_c(self, c):
        """niwqg/QGModel.py:522-534."""
        c = np.asarray(c)
        if np.iscomplexobj(c):
            raise TypeError("set_c needs a real array (numpy.fft.rfft2 rejects complex input)")
        self._h.set_c(c)

    def save_checkpoint(self, path):
        """See Kernel.save_checkpoint."""
        Checkpoint.save(self, path)

    def load_checkpoint(self, path):
        """See Kernel.load_checkpoint."""
        Checkpoint.load(self, path)

    @classmethod
    def from_checkpoint(cls, path, **overrides):
        """See Kernel.from_checkpoint."""
        return Checkpoint.from_checkpoint(cls, path, **overrides)

    def _invert(self):
        """niwqg/QGModel.py:497-505: ph = -wv2i*qh is maintained on the device; nothing to do."""
        return None

    def _print_status(self):
        """niwqg/QGModel.py:554-575."""
        self.tc += 1
        self.t += self.dt
        if (self.tc % self.twrite) == 0:
            st = self._h.status()
            s = st[int(np.argmax(st[:, 3]))]
            self.ke = float(st[0, 0]) if self.batch == 1 else st[:, 0]
            self.cfl = float(st[0, 3]) if self.batch == 1 else st[:, 3]
            self.logger.info('Step: %i, Time: %4.3e, P: %4.3e , Ke: %4.3e, CFL: %4.3f',
                             self.tc, self.t, self.t / self.tmax, s[0], s[3])
            assert np.all(st[:, 3] < self.cflmax), self.logger.error('CFL condition violated')

    def jacobian_psi_q(self):
        """niwqg/QGModel.py:469-481 (half-spectrum array)."""
        return self._h.jacobian(nat.JAC_PSI_Q)

    def spec_var(self, ph):
        """niwqg/QGModel.py:611-619 (host array in rfft2 layout)."""
        var_dens = 2. * np.abs(ph) ** 2 / self.M ** 2
        var_dens[:, 0] *= 0.5
        var_dens[:, -1] *= 0.5
        var_dens[0, 0] = 0
        return var_dens.sum()

    def _calc_ke_qg(self):
        st = self._h.status()
        return float(st[0, 0]) if self.batch == 1 else st[:, 0]

    def _calc_cfl(self):
        st = self._h.status()
        return float(st[0, 3]) if self.batch == 1 else st[:, 3]

    # ------------------------------------------------------------ diagnostics
    def _calc_derived_fields(self):
        d = self._h.scalars("diagnostics")
        self._diag = d[0] if self.batch == 1 else d.T
        S = nat.S
        self.C2, self.gradC2, self.Gamma_c = self._diag[S["C2"]], self._diag[S["GRADC2"]], self._diag[S["GAMMA_C"]]

    def _initialize_diagnostics(self):
        """Registry of niwqg/QGModel.py:632-722, same order."""
        S = nat.S
        self.diagnostics = dict()
        reg = [('time', 'Time', 'seconds', lambda self: self.t),
               ('ke_qg', 'Quasigeostrophic Kinetic Energy', r'm^2 s^{-2}', lambda self: self._diag[S["KE_QG"]]),
               ('Ke', 'Quasigeostrophic Kinetic Energy, from energy equation', r'm^2 s^{-2}',
                lambda self: self._diag[S["KE"]]),
               ('ens', 'Quasigeostrophic Potential Enstrophy', r's^{-2}', lambda self: self._diag[S["ENS"]]),
               ('ep_psi', 'The hyperviscous dissipation of QG kinetic energy', r'$m^2 s^{-3}$',
                lambda self: self._diag[S["EP_PSI"]]),
               ('chi_q', 'The hyperviscous dissipation of QG kinetic energy', r'$s^{-3}$',
                lambda self: self._diag[S["CHI_Q"]]),
               ('C2', 'Passive tracer variance', r'[scalar]^2', lambda self: self._diag[S["C2"]]),
               ('cvar', 'Passive tracer variance, from variance equation', r'[scalar]^2',
                lambda self: self._diag[S["CVAR"]]),
               ('gradC2', 'Gradient of Passive tracer variance', r'[scalar]^2 / m^2', lambda self: self._diag[S["GRADC2"]]),
               ('Gamma_c', 'Rate of generation of passive tracer gradient variance', r'[scalar]^2 / (m^2 s)',
                lambda self: self._diag[S["GAMMA_C"]]),
               ('ep_c', 'The dissipation of tracer variance', r'$s^{-3}$', lambda self: self._diag[S["EP_C"]]),
               ('chi_c', 'The dissipation of tracer gradient variance', r'$s^{-3}$', lambda self: self._diag[S["CHI_C"]])]
        for name, desc, units, fn in reg:
            add_diagnostic(self, name, description=desc, units=units, types='scalar', function=fn)
