"""Host side of the NIW-QG kernel family with the reference's class protocol
(niwqg/Kernel.py): same constructor keywords, ``set_q`` / ``set_phi`` / ``run`` /
``run_with_snapshots`` / ``_step_forward`` / ``_step_etdrk4``, the same attribute
names and diagnostics dictionary.  All arithmetic on grid-sized arrays happens in
the CUDA library behind the C ABI (include/niwqg_b200.h); attribute reads copy the
field back from the device on demand.
"""
import logging

import numpy as np
from numpy import pi

from . import _native as nat
from . import Checkpoint
from .Particles import Particles
from .Diagnostics import add_diagnostic, increment_diagnostics, get_diagnostic, describe_diagnostics  # noqa: F401
from .Saving import initialize_save_snapshots, save_setup, save_snapshots, save_diagnostics


class _DeviceField(object):
    """Read-only attribute backed by a device field (Seam 3, SURVEY.md section 8b)."""

    def __init__(self, name):
        self.name = name

    def __get__(self, obj, objtype=None):
        if obj is None:
            return self
        return obj._h.field(self.name)


class _Scalar(object):
    """Integrated budget kept on the device (Ke, Pw, Kw).  Read-only: the reference lets user code assign to it, which
    here would silently shadow the device value, so an assignment raises instead."""

    def __init__(self, name):
        self.name = name

    def __get__(self, obj, objtype=None):
        if obj is None:
            return self
        v = obj._h.scalars()[:, nat.S[self.name]]
        return float(v[0]) if obj.batch == 1 else v

    def __set__(self, obj, value):
        raise AttributeError("%s lives on the device (set it through set_q / set_phi)" % self.name)


class _LazyGrid(object):
    """Whole-grid host array of the reference's grid set-up (niwqg/Kernel.py:232-265), built on first use and cached.
    The device never reads these (wavenumbers are recomputed from indices in the kernels), and at 8192^2 the ten of them
    are 6 GB of host memory and most of the model construction time."""

    def __init__(self, name, build):
        self.name, self.build = name, build

    def __get__(self, obj, objtype=None):
        if obj is None:
            return self
        v = self.build(obj)
        obj.__dict__[self.name] = v        # non-data descriptor: the instance attribute wins from now on
        return v


def _wv2i(self):
    out = np.zeros_like(self.wv2)
    nz = self.wv2 != 0.
    out[nz] = self.wv2[nz] ** -1
    return out


class Kernel(Particles):
    """Doubly periodic single-vertical-mode NIW + barotropic QG pseudo-spectral kernel.

    Parameters are those of niwqg/Kernel.py:70-98 (SI units), plus
        batch  : number of independent ensemble members stepped together (default 1)
    With batch > 1, each of U, f, N, m, nu, nu4, mu, nuw, nu4w, muw may be a sequence of batch values, one per member
    (a parameter sweep in one batch; kappa, kappa2 and hslash are then arrays too).  nx, L, dt, use_filter, dealias
    and g are common to all members.
        device : CUDA device ordinal (default 0)
        rank, nranks, nccl_id : slab decomposition of ONE grid over nranks GPUs (one process per GPU;
                 see niwqg_b200/slab.py).  set_q/set_phi then take the whole-grid array (each rank keeps its
                 rows) or the rank's rows; physical attributes return the rank's rows.
    ``use_mkl`` / ``nthreads`` are accepted and ignored (the FFT backend is the CUDA engine).
    """

    _model_id = None     # set by subclasses
    _ke = None
    # constructor keywords a checkpoint records: the ones that reach the arithmetic (a restore requires them unchanged)
    # and the ones that set the cadence and output of a run (from_checkpoint takes them over unless overridden)
    _checkpoint_params = ("L", "dt", "U", "f", "N", "m", "g", "nu4", "nu4w", "nu", "nuw", "mu", "muw", "use_filter",
                          "dealias")
    _checkpoint_run = ("twrite", "tmax", "cflmax", "tdiags", "tsave_snapshots", "save_to_disk", "overwrite", "path")
    _checkpoint_attr = {"tsave_snapshots": "tsnaps"}

    # device-backed attributes (names of the reference's numpy arrays)
    q = _DeviceField("Q"); qh = _DeviceField("QH"); p = _DeviceField("P"); ph = _DeviceField("PH")
    phi = _DeviceField("PHI"); phih = _DeviceField("PHIH")
    phix = _DeviceField("PHIX"); phiy = _DeviceField("PHIY"); lapphi = _DeviceField("LAPPHI")
    u = _DeviceField("U"); v = _DeviceField("V"); q_psi = _DeviceField("QPSI")
    filtr = _DeviceField("FILTR")
    expch = _DeviceField("EXPCH"); expch_h = _DeviceField("EXPCH_H"); Qh = _DeviceField("QHCOEF")
    f0 = _DeviceField("F0"); fab = _DeviceField("FAB"); fc = _DeviceField("FC")
    expchw = _DeviceField("EXPCHW"); expch_hw = _DeviceField("EXPCH_HW"); Qhw = _DeviceField("QHWCOEF")
    f0w = _DeviceField("F0W"); fabw = _DeviceField("FABW"); fcw = _DeviceField("FCW")
    Ke = _Scalar("KE"); Pw = _Scalar("PW"); Kw = _Scalar("KW")
    # whole-grid host arrays, on demand
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

    def __init__(self, nx=128, ny=None, L=5e5, dt=10000., twrite=1000., tmax=250000., use_filter=True,
                 cflmax=0.8, U=.0, f=1.e-4, N=0.01, m=0.025, g=9.81, nu4=0, nu4w=0, nu=20, nuw=50., mu=0, muw=0,
                 dealias=False, save_to_disk=False, overwrite=True, tsave_snapshots=10, tdiags=10,
                 path='output/', use_mkl=False, nthreads=1, batch=1, device=0, rank=0, nranks=1,
                 nccl_id=None):
        kw = nat.member_keywords(batch, dict(U=U, f=f, N=N, m=m, nu=nu, nu4=nu4, mu=mu, nuw=nuw, nu4w=nu4w, muw=muw),
                                 dict(nx=nx, L=L, dt=dt, use_filter=use_filter, dealias=dealias, g=g))
        U, f, N, m, nu, nu4, mu, nuw, nu4w, muw = (kw[k] for k in ("U", "f", "N", "m", "nu", "nu4", "mu", "nuw", "nu4w",
                                                                   "muw"))
        self.nx = nx
        self.ny = nx                    # niwqg/Kernel.py:100-103: ny is ignored (F9)
        self.L = L
        self.W = L
        self.dt = dt
        self.twrite = twrite
        self.tmax = tmax
        self.dealias = dealias
        self.U = U
        self.g = g
        self.nu4, self.nu4w, self.nu, self.nuw, self.mu, self.muw = nu4, nu4w, nu, nuw, mu, muw
        self.f, self.N, self.m = f, N, m
        self.kappa = self.m * self.f / self.N
        self.kappa2 = self.kappa ** 2
        self.cflmax = cflmax
        self.hslash = self.f / self.kappa2
        self.save_to_disk = save_to_disk
        self.overwrite = overwrite
        self.tsnaps = tsave_snapshots
        self.tdiags = tdiags
        self.path = path
        self.use_filter = use_filter
        self.use_mkl = use_mkl
        self.nthreads = nthreads
        self.batch = batch
        self.device = device
        # slab decomposition of this grid over nranks GPUs, one process per GPU (niwqg_b200/slab.py builds these)
        self.rank, self.nranks, self._nccl_id = rank, nranks, nccl_id
        if save_to_disk and nranks > 1:
            # every rank would write its own rows under the same file names (niwqg/Saving.py has no notion of ranks)
            raise NotImplementedError("save_to_disk with a slab-decomposed grid: gather with niwqg_b200.slab.gather_rows "
                                      "and write from one rank")

        self._initialize_logger()
        self.logger.info(self.model)
        self._initialize_grid()
        self._create_backend()           # allocation, filter and ETDRK4 tables live on the device
        self._initialize_time()
        initialize_save_snapshots(self, self.path)
        save_setup(self, )
        self._initialize_fft()
        self._initialize_diagnostics()

    # ------------------------------------------------------------------ set-up
    def _create_backend(self):
        self._h = nat.Handle(model=self._model_id, nx=self.nx, batch=self.batch, device=self.device,
                             L=self.L, dt=self.dt, U=self.U, f=self.f, N=self.N, m=self.m,
                             nu=self.nu, nu4=self.nu4, mu=self.mu, nuw=self.nuw, nu4w=self.nu4w, muw=self.muw,
                             beta=0.0, use_filter=int(bool(self.use_filter)), dealias=int(bool(self.dealias)),
                             passive_scalar=0, nu4c=0.0, nuc=0.0, muc=0.0,
                             **({} if self.nranks <= 1 else dict(rank=self.rank, nranks=self.nranks,
                                                                  nccl_id=self._nccl_id)))
        if self.use_filter:
            self.logger.info(' Using filter')
        elif self.dealias:
            self.logger.info(' Dealiasing with 2/3 rule')
        else:
            self.logger.info(' No dealiasing; no filter')

    def _initialize_time(self):
        self.t = 0
        self.tc = 0

    def _initialize_grid(self):
        """Scalars and 1-D arrays of niwqg/Kernel.py:227-265; the 2-D arrays (x, y, k, l, ik, il, wv2, wv, wv4, wv2i)
        are lazy class attributes (_LazyGrid)."""
        self.dk = 2. * pi / self.L
        self.dl = 2. * pi / self.L
        self.nl = self.ny
        self.nk = self.nl
        self.ll = self.dl * np.append(np.arange(0., self.nx / 2), np.arange(-self.nx / 2, 0.))
        self.kk = self.ll.copy()
        self.dx = self.L / self.nx
        self.dy = self.W / self.ny
        self.M = self.nx * self.ny

    def _initialize_logger(self):
        """niwqg/Kernel.py:286-304."""
        self.logger = logging.getLogger(__name__)
        fhandler = logging.StreamHandler()
        fhandler.setFormatter(logging.Formatter('%(levelname)s: %(message)s'))
        if not self.logger.handlers:
            self.logger.addHandler(fhandler)
        self.logger.setLevel(10)
        self.logger.propagate = False
        self.logger.info(' Logger initialized')

    def _initialize_fft(self):
        """The FFT backend seam (niwqg/Kernel.py:553-566): callables on N x N host arrays,
        numpy conventions, executed by the CUDA engine."""
        def _fft(x):
            x = np.asarray(x)
            if np.iscomplexobj(x):
                return self._h.fft2(x, nat.FFT_C2C_FWD)
            return self._h.fft2(x, nat.FFT_R2C_FULL)

        self.fft = _fft
        self.ifft = lambda x: self._h.fft2(x, nat.FFT_C2C_INV)

    # ------------------------------------------------------------------ driver
    def run_with_snapshots(self, tsnapstart=0., tsnapint=432000.):
        """niwqg/Kernel.py:161-181."""
        tsnapints = np.ceil(tsnapint / self.dt)
        while (self.t < self.tmax):
            self._step_forward()
            if self.t >= tsnapstart and (self.tc % tsnapints) == 0:
                yield self.t
        return

    def run(self):
        """niwqg/Kernel.py:183-203."""
        if self.save_to_disk:
            save_snapshots(self, fields=['t', 'q', 'phi'])
        while (self.t < self.tmax):
            self._step_forward()
        if self.save_to_disk:
            save_diagnostics(self)

    def _step_forward(self):
        """niwqg/Kernel.py:205-217."""
        self._step_etdrk4()
        increment_diagnostics(self, )
        self._print_status()
        save_snapshots(self, fields=['t', 'q', 'phi'])

    def _step_etdrk4(self):
        """One ETDRK4 step on the device (niwqg/Kernel.py:307-397; YBJModel.py:52-87)."""
        self._h.step(1)

    def step(self, nsteps=1):
        """nsteps device steps back to back, without host-side diagnostics (clock is advanced)."""
        self._h.step(nsteps)
        for _ in range(int(nsteps)):
            self.tc += 1
            self.t += self.dt

    # ---------------------------------------------------------------- seeding
    def set_q(self, q=None):
        """niwqg/Kernel.py:520-535 (inverts with the current phi, F5).  ``self.ke = Ke`` of the reference is served on
        first read (property below): reading it here would make the host wait for the inversion, which otherwise runs
        on the device while the caller already uploads phi.  ``q=None`` (extension): seed from the array queued with
        ``stage_inputs``."""
        self._h.set_q(q)
        self._ke = None

    def stage_inputs(self, q=None, phi=None):
        """Extension (no reference counterpart): start the host-to-device copy of the NEXT ``set_q()`` / ``set_phi()``
        arguments now, on the copy stream, and return at once - the copy then overlaps the steps in between.  The
        arrays (pinned host memory for a truly asynchronous copy) must stay unchanged until ``set_q()`` / ``set_phi()``
        - called without an argument - have consumed them."""
        if q is not None:
            self._h.stage_q(q)
        if phi is not None:
            self._h.stage_phi(phi)

    @property
    def ke(self):
        if self._ke is None:
            self._ke = self.Ke
        return self._ke

    @ke.setter
    def ke(self, value):
        self._ke = value

    def set_phi(self, phi=None):
        """niwqg/Kernel.py:538-551 (does not re-invert, F5).  ``phi=None``: the array queued with ``stage_inputs``."""
        self._h.set_phi(phi)

    # ------------------------------------------------------------ checkpoint
    def save_checkpoint(self, path, dist=None):
        """Write the model's complete state to the directory ``path`` (niwqg_b200/Checkpoint.py): every carried device
        field, Ke/Pw/Kw and the other scalars a step carries, t, tc, the diagnostics and the status attributes.  Changes
        nothing on the model.  ``path`` must be new, empty or a checkpoint: another directory is never replaced.  Slab
        runs call it on every rank (``dist``: torch.distributed, default the global one; an error on any rank is raised
        on every rank)."""
        Checkpoint.save(self, path, dist)

    def load_checkpoint(self, path, dist=None):
        """Restore a checkpoint written by ``save_checkpoint`` from a model of the same class, nx, batch and arithmetic
        parameters (ValueError names any difference; the model is left as it was).  The steps that follow are
        bit-for-bit those of the saved run; on another layout (slab ranks, split transforms) they agree to rounding.
        ``dist`` as for save_checkpoint."""
        Checkpoint.load(self, path, dist)

    @classmethod
    def from_checkpoint(cls, path, **overrides):
        """The model saved in ``path``, built from its saved keywords and restored.  ``overrides`` replace keywords,
        e.g. tmax, tdiags, path, device (or rank/nranks/nccl_id through slab.make_model).  Overriding an arithmetic
        parameter such as dt or a dissipation coefficient is allowed, with a warning: the run then no longer continues
        the saved one exactly."""
        return Checkpoint.from_checkpoint(cls, path, **overrides)

    # ---------------------------------------------------------------- status
    def _print_status(self):
        """niwqg/Kernel.py:568-598."""
        self.tc += 1
        self.t += self.dt
        if (self.tc % self.twrite) == 0:
            st = self._h.status()
            pick = (lambda j: float(st[0, j])) if self.batch == 1 else (lambda j: st[:, j])
            self.ke, self.kew, self.pew, self.cfl = pick(0), pick(1), pick(2), pick(3)
            s = st[int(np.argmax(st[:, 3]))]
            self.logger.info('Step: %4i, Time: %2.1e, P: %2.1e, Ke: %4.3e, Kw: %4.3e, Pw: %4.3e, CFL: %3.2f',
                             self.tc, self.t, self.t / self.tmax, s[0], s[1], s[2], s[3])
            assert np.all(st[:, 3] < self.cflmax), self.logger.error('CFL condition violated')

    # ------------------------------------------------- attribute-level methods
    def jacobian_psi_q(self):
        """niwqg/Kernel.py:471-486."""
        return self._h.jacobian(nat.JAC_PSI_Q)

    def jacobian_psi_phi(self):
        """niwqg/Kernel.py:457-469 (YBJModel.py:123-133 / QLModel.py:65-67 variants on the device)."""
        return self._h.jacobian(nat.JAC_PSI_PHI)

    def spec_var(self, ph):
        """Variance from a full c2c spectrum held on the host (niwqg/Kernel.py:654-658)."""
        var_dens = np.abs(ph) ** 2 / self.M ** 2
        var_dens[0, 0] = 0.
        return var_dens.sum()

    def _status_value(self, j):
        st = self._h.status()
        return float(st[0, j]) if self.batch == 1 else st[:, j]

    def _calc_ke_qg(self):
        return self._status_value(0)

    def _calc_ke_niw(self):
        return self._status_value(1)

    def _calc_pe_niw(self):
        return self._status_value(2)      # refreshes phix, phiy on the device (F6)

    def _calc_cfl(self):
        return self._status_value(3)

    # -------------------------------- the reference's per-quantity helpers (user scripts call them directly)
    def _invert(self):
        """niwqg/Kernel.py:488-490 hook: the inversion runs on the device inside set_q and every stage; the carried
        fields (ph, q, qw, u, v) are always consistent with qh, so there is nothing left to do here."""

    def _calc_rel_vorticity(self):
        """niwqg/Kernel.py:492-501 / CoupledModel.py:145-152: q_psi is carried on the device (attribute ``q_psi``)."""

    def _diag_slot(self, name):
        d = self._h.scalars("diagnostics")
        v = d[:, nat.S[name]]
        return float(v[0]) if self.batch == 1 else v

    def _calc_energy_conversion(self):
        """niwqg/Kernel.py:664-701: gamma1, gamma2, xi1, xi2, pi of the current state."""
        self._calc_derived_fields()

    def _calc_icke_niw(self):
        """niwqg/Kernel.py:703-706."""
        self._calc_derived_fields()

    def _calc_conc(self):
        return self._diag_slot("CONC")

    def _calc_skewness(self):
        return self._diag_slot("SKEW")

    def _calc_ens(self):
        return self._diag_slot("ENS")

    def _calc_ep_phi(self):
        return self._diag_slot("EP_PHI")

    def _calc_ep_psi(self):
        return self._diag_slot("EP_PSI")

    def _calc_chi_q(self):
        return self._diag_slot("CHI_Q")

    def _calc_chi_phi(self):
        return self._diag_slot("CHI_PHI")

    def _calc_strain(self):
        """niwqg/Kernel.py:503-509: geostrophic rate of strain from the device ph (three transforms on the CUDA engine)."""
        ph = self.ph
        pxx, pyy = self.ifft(-self.k * self.k * ph).real, self.ifft(-self.l * self.l * ph).real
        pxy = self.ifft(-self.k * self.l * ph).real
        self.qg_strain = 4 * (pxy ** 2) + (pxx - pyy) ** 2

    def _calc_OW(self):
        """niwqg/Kernel.py:511-518: Okubo-Weiss parameter."""
        self._calc_strain()
        return self.qg_strain ** 2 - self.q_psi ** 2

    # ------------------------------------------------------------ diagnostics
    def _calc_derived_fields(self):
        """niwqg/Kernel.py:870-878: one device pass evaluates every registered scalar."""
        d = self._h.scalars("diagnostics")
        self._diag = d[0] if self.batch == 1 else d.T
        S = nat.S
        self.gamma1, self.gamma2 = self._diag[S["GAMMA1"]], self._diag[S["GAMMA2"]]
        self.xi1, self.xi2, self.pi = self._diag[S["XI1"]], self._diag[S["XI2"]], self._diag[S["PI"]]
        self.ke_niw, self.cke_niw, self.ike_niw = (self._diag[S["KE_NIW"]], self._diag[S["CKE_NIW"]],
                                                   self._diag[S["IKE_NIW"]])
        self._calc_class_derived_fields()

    def _calc_class_derived_fields(self):
        pass

    def _initialize_class_diagnostics(self):
        pass

    def _initialize_diagnostics(self):
        """niwqg/Kernel.py:708-716."""
        self.diagnostics = dict()
        self._initialize_kernel_diagnostics()
        self._initialize_class_diagnostics()

    def _initialize_kernel_diagnostics(self):
        """Registry of niwqg/Kernel.py:718-868, in the same order."""
        S = nat.S
        reg = [
            ('time', 'Time', 'seconds', lambda self: self.t),
            ('Ke', 'Quasigeostrophic Kinetic Energy, from energy equation', r'm^2 s^{-2}', lambda self: self._diag[S["KE"]]),
            ('Pw', 'NIW Potential Energy, from energy equation', r'm^2 s^{-2}', lambda self: self._diag[S["PW"]]),
            ('Kw', 'NIW Kinetic Energy, from energy equation', r'm^2 s^{-2}', lambda self: self._diag[S["KW"]]),
            ('ke_qg', 'Quasigeostrophic Kinetic Energy', r'm^2 s^{-2}', lambda self: self._diag[S["KE_QG"]]),
            ('ens', 'Quasigeostrophic Potential Enstrophy', r's^{-2}', lambda self: self._diag[S["ENS"]]),
            ('ke_niw', 'Near-inertial Kinetic Energy', r'm^2 s^{-2}', lambda self: self._diag[S["KE_NIW"]]),
            ('cke_niw', 'Kinetic Energy of Laterally Coherent Near-Inertial Waves', r'm^2 s^{-2}',
             lambda self: self._diag[S["CKE_NIW"]]),
            ('ike_niw', 'Kinetic Energy of Laterally Incoherent Near-Inertial Waves', r'm^2 s^{-2}',
             lambda self: self._diag[S["IKE_NIW"]]),
            ('pe_niw', 'Near-inertial Potential Energy', r'm^2 s^{-2}', lambda self: self._diag[S["PE_NIW"]]),
            ('conc_niw', 'Correlation between relative vorticity and near-inertial KE', r'unitless',
             lambda self: self._diag[S["CONC"]]),
            ('skew', 'Skewness', r'unitless', lambda self: self._diag[S["SKEW"]]),
            ('gamma_r', 'The energy conversion due to refraction', r'$m^2 s^{-3}$', lambda self: self._diag[S["GAMMA1"]]),
            ('gamma_a', 'The energy conversion due to advection', r'$m^2 s^{-3}$', lambda self: self._diag[S["GAMMA2"]]),
            ('xi_r', 'The QG energy generation due to wave dissipation, vorticity', r'$m^2 s^{-3}$',
             lambda self: self._diag[S["XI1"]]),
            ('xi_a', 'The QG energy generation due to wave dissipation, advection', r'$m^2 s^{-3}$',
             lambda self: self._diag[S["XI2"]]),
            ('pi', 'The NIW kinetic energy conversion from coherent to incoherent', r'$m^2 s^{-3}$',
             lambda self: self._diag[S["PI"]]),
            ('ep_phi', 'The hyperviscous dissipation of NIW kinetic energy', r'$m^2 s^{-3}$',
             lambda self: self._diag[S["EP_PHI"]]),
            ('ep_psi', 'The hyperviscous dissipation of QG kinetic energy', r'$m^2 s^{-3}$',
             lambda self: self._diag[S["EP_PSI"]]),
            ('chi_q', 'The hyperviscous dissipation of QG kinetic energy', r'$s^{-3}$', lambda self: self._diag[S["CHI_Q"]]),
            ('chi_phi', 'The hyperviscous dissipation of NIW potential energy', r'$s^{-3}$',
             lambda self: self._diag[S["CHI_PHI"]]),
        ]
        for name, desc, units, fn in reg:
            add_diagnostic(self, name, description=desc, units=units, types='scalar', function=fn)
