"""CPU oracle for the niwqg ETDRK4 hot path  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module.  The product path
(``niwqg_b200``) never does: it fails loudly when the CUDA library is missing.

What this is
------------
A numpy restatement of the reference solver's arithmetic for the path named by
BASELINE.json (SURVEY.md section 8a): the ETDRK4 step of the NIW-QG kernel
family (Coupled / UnCoupled / YBJ / repaired-QL) and of the stand-alone QG
model, the inversions, Jacobians, energy-budget terms and the diagnostics tick
that feeds back into the step.  It is organised differently from the reference
(one state class, table-driven model variants, row-chunked coefficient
generation so 4096^2+ initialises in bounded memory), but every floating point
operation is issued in the same order as the reference issues it, so results
are bit-identical to the reference on the same numpy.  Each method cites the
reference lines it follows (paths relative to the reference checkout).

Pinning
-------
Parity is PINNED: ``tests/golden/make_golden.py`` imports the unmodified
reference from a checkout of it (with an ``h5py`` import stub) and stores its
outputs under ``tests/golden/*.npz``; ``tests/test_oracle_cpu.py`` checks this
oracle against those vectors bit-for-bit.

Third-party arithmetic the reference relies on: ``numpy.fft`` (pocketfft,
numpy>=1.8 per requirements.txt:1, 2.3.5 installed) - called here through the
same four entry points.
"""
import numpy as np

_TWO_PI = 2.0 * np.pi

MODELS = ("coupled", "uncoupled", "ybj", "ql")


def etdrk4_tables(ch, dt, rows_per_chunk=None):
    """Kassam-Trefethen contour-mean ETDRK4 coefficients for exponent ``ch=c*dt``.

    Follows niwqg/Kernel.py:424-433 (same for :448-454, YBJModel.py:98-121,
    QGModel.py:434-443): 32 roots of unity r_j=exp(2 pi i j/32), j=1..32,
    LR=ch+r_j, means over j.  Evaluated in row chunks (the reference builds one
    (N,N,32) temporary, F12 in SURVEY.md) - per-element arithmetic and the
    reduction over the contiguous last axis are unchanged, so the values are
    bit-identical.
    Returns (E, E2, Q, f0, fab, fc).
    """
    M = 32
    r = 1.0 * np.exp(2j * np.pi * ((np.arange(1.0, M + 1)) / M))
    E = np.exp(ch)
    E2 = np.exp(ch / 2.0)
    Q = np.empty_like(ch)
    f0 = np.empty_like(ch)
    fab = np.empty_like(ch)
    fc = np.empty_like(ch)
    n = ch.shape[0]
    if rows_per_chunk is None:
        rows_per_chunk = max(1, min(n, (1 << 22) // max(1, ch.shape[1] * M)))
    for a in range(0, n, rows_per_chunk):
        b = min(n, a + rows_per_chunk)
        LR = ch[a:b, :, np.newaxis] + r[np.newaxis, np.newaxis, :]
        LR2 = LR * LR
        LR3 = LR2 * LR
        Q[a:b] = dt * (((np.exp(LR / 2.0) - 1.0) / LR).mean(axis=-1))
        f0[a:b] = dt * (((-4.0 - LR + (np.exp(LR) * (4.0 - 3.0 * LR + LR2))) / LR3).mean(axis=-1))
        fab[a:b] = dt * (((2.0 + LR + np.exp(LR) * (-2.0 + LR)) / LR3).mean(axis=-1))
        fc[a:b] = dt * (((-4.0 - 3.0 * LR - LR2 + np.exp(LR) * (4.0 - LR)) / LR3).mean(axis=-1))
    return E, E2, Q, f0, fab, fc


def spectral_filter(k, l, dx, dy, use_filter, dealias, nx, ny, int_slices=True):
    """Exponential filter / 2-3 mask / ones.  niwqg/Kernel.py:267-284."""
    if use_filter:
        cphi = 0.65 * np.pi
        wvx = np.sqrt((k * dx) ** 2.0 + (l * dy) ** 2.0)
        filtr = np.exp(-23.6 * (wvx - cphi) ** 4.0)
        filtr[wvx <= cphi] = 1.0
    elif dealias:
        filtr = np.ones_like(k)
        filtr[nx // 3:2 * nx // 3, :] = 0.0
        filtr[:, ny // 3:2 * ny // 3] = 0.0
    else:
        filtr = np.ones_like(k)
    return filtr


class NIWQGOracle(object):
    """Kernel-family oracle (complex c2c transforms).

    model: 'coupled' (niwqg/CoupledModel.py), 'uncoupled' (niwqg/UnCoupledModel.py),
           'ybj' (niwqg/YBJModel.py) or 'ql' (repaired QL: CoupledModel with the
           wave advection of niwqg/QLModel.py:65-67, see SURVEY.md section 8c).
    Constructor keywords and defaults: niwqg/Kernel.py:70-98.
    """

    def __init__(self, model="coupled", nx=128, ny=None, L=5e5, dt=10000., twrite=1000.,
                 tmax=250000., use_filter=True, cflmax=0.8, U=.0, f=1.e-4, N=0.01,
                 m=0.025, g=9.81, nu4=0, nu4w=0, nu=20, nuw=50., mu=0, muw=0,
                 dealias=False, tdiags=10):
        assert model in MODELS
        self.model = model
        self.nx = nx
        self.ny = nx                       # Kernel.py:100-103 (ny ignored, F9)
        self.L = self.W = L
        self.dt, self.twrite, self.tmax = dt, twrite, tmax
        self.U, self.g = U, g
        self.nu4, self.nu4w, self.nu, self.nuw, self.mu, self.muw = nu4, nu4w, nu, nuw, mu, muw
        self.f, self.N, self.m = f, N, m
        self.kappa = self.m * self.f / self.N       # Kernel.py:121-125
        self.kappa2 = self.kappa ** 2
        self.hslash = self.f / self.kappa2
        self.cflmax = cflmax
        self.use_filter, self.dealias, self.tdiags = use_filter, dealias, tdiags
        self._grid()
        self._alloc()
        self.filtr = spectral_filter(self.k, self.l, self.dx, self.dy, use_filter,
                                     dealias, self.nx, self.ny)
        self._coefficients()
        self.t = 0
        self.tc = 0
        self.fft = lambda x: np.fft.fft2(x)         # Kernel.py:565-566
        self.ifft = lambda x: np.fft.ifft2(x)
        self.diag = {}                              # name -> list of scalars

    # ------------------------------------------------------------------ setup
    def _grid(self):
        """niwqg/Kernel.py:227-265."""
        nx, ny, L = self.nx, self.ny, self.L
        self.x, self.y = np.meshgrid(np.arange(0.5, nx, 1.) / nx * L,
                                     np.arange(0.5, ny, 1.) / ny * self.W)
        self.dk = self.dl = 2. * np.pi / L
        self.nl = ny
        self.nk = self.nl
        self.ll = self.dl * np.append(np.arange(0., nx / 2), np.arange(-nx / 2, 0.))
        self.kk = self.ll.copy()
        self.k, self.l = np.meshgrid(self.kk, self.ll)
        self.ik = 1j * self.k
        self.il = 1j * self.l
        self.dx = L / nx
        self.dy = self.W / ny
        self.M = nx * ny
        self.wv2 = self.k ** 2 + self.l ** 2
        self.wv = np.sqrt(self.wv2)
        self.wv4 = self.wv2 ** 2
        nz = self.wv2 != 0.
        self.wv2i = np.zeros_like(self.wv2)
        self.wv2i[nz] = self.wv2[nz] ** -1

    def _alloc(self):
        """niwqg/CoupledModel.py:33-55 (identical in the other subclasses)."""
        shp = (self.ny, self.nx)
        self.q = np.zeros(shp, np.float64)
        self.qh = np.zeros(shp, np.complex128)
        self.p = np.zeros(shp, np.float64)
        self.ph = np.zeros(shp, np.complex128)
        self.phi = np.zeros(shp, np.complex128)
        self.phih = np.zeros(shp, np.complex128)

    def _coefficients(self):
        """niwqg/Kernel.py:400-454; YBJ builds the wave set only (YBJModel.py:89-121)."""
        z = np.zeros((self.nl, self.nk), np.complex128)
        if self.model != "ybj":
            c = z - 1j * self.k * self.U
            c += -self.nu4 * self.wv4 - self.nu * self.wv2 - self.mu
            ch = c * self.dt
            (self.expch, self.expch_h, self.Qh, self.f0, self.fab, self.fc) = \
                etdrk4_tables(ch, self.dt)
        c = z - 1j * self.k * self.U
        c += -self.nu4w * self.wv4 - 0.5j * self.f * (self.wv2 / self.kappa2) \
            - self.nuw * self.wv2 - self.muw
        ch = c * self.dt
        (self.expchw, self.expch_hw, self.Qhw, self.f0w, self.fabw, self.fcw) = \
            etdrk4_tables(ch, self.dt)

    # -------------------------------------------------------------- seeding
    def set_q(self, q):
        """niwqg/Kernel.py:520-535 (inverts with whatever phi is current, F5)."""
        self.q = q
        self.qh = self.fft(self.q)
        self._invert()
        self._rel_vorticity()
        self.u, self.v = self.ifft(-self.il * self.ph).real, self.ifft(self.ik * self.ph).real
        self.Ke = self.ke = self.ke_qg()

    def set_phi(self, phi):
        """niwqg/Kernel.py:538-551 (does not re-invert, F5)."""
        self.phi = phi
        self.phih = self.fft(self.phi)
        self.Pw = self.pe_niw()
        self.Kw = self.ke_niw()

    # ------------------------------------------------------------ inversion
    def jacobian_phic_phi(self):
        """niwqg/CoupledModel.py:59-73."""
        self.phix, self.phiy = self.ifft(self.ik * self.phih), self.ifft(self.il * self.phih)
        jach = self.fft((1j * (np.conj(self.phix) * self.phiy - np.conj(self.phiy) * self.phix)).real)
        jach[0, 0] = 0
        return jach

    def _invert(self):
        if self.model in ("coupled", "ql"):
            # niwqg/CoupledModel.py:75-97
            self.phi2 = np.abs(self.phi) ** 2
            self.gphi2h = -self.wv2 * self.fft(self.phi2)
            self.qwh = 0.5 * (0.5 * self.gphi2h + self.jacobian_phic_phi()) / self.f
            self.qwh *= self.filtr
            self.pw = self.ifft((self.wv2i * self.qwh)).real
            self.pv = self.ifft(-(self.wv2i * self.qh)).real
            self.p = self.pv + self.pw
            self.ph = self.fft(self.p)
            self.q = self.ifft(self.qh).real
        elif self.model == "uncoupled":
            # niwqg/UnCoupledModel.py:54-64
            self.p = self.ifft(-(self.wv2i * self.qh)).real
            self.ph = self.fft(self.p)
            self.q = self.ifft(self.qh).real
        else:
            # niwqg/YBJModel.py:141-146
            self.ph = -self.wv2i * self.qh

    def _rel_vorticity(self):
        if self.model in ("coupled", "ql"):
            # niwqg/CoupledModel.py:145-152
            self.qw = self.ifft(self.qwh).real
            self.q_psi = (self.q - self.qw)
        else:
            # niwqg/Kernel.py:492-501
            self.q_psi = (self.q)

    # ------------------------------------------------------------ jacobians
    def jacobian_psi_q(self):
        """niwqg/Kernel.py:471-486."""
        self.u, self.v = self.ifft(-self.il * self.ph).real, self.ifft(self.ik * self.ph).real
        q = self.ifft(self.qh).real
        jach = self.ik * self.fft(self.u * q) + self.il * self.fft(self.v * q)
        jach[0, 0] = 0
        return jach

    def jacobian_psi_phi(self):
        if self.model == "ql":
            # niwqg/QLModel.py:65-67 on top of CoupledModel (repaired QL)
            self.ph_q = -self.wv2i * self.qh
            self.uq, self.vq = self.ifft(-self.il * self.ph_q).real, self.ifft(self.ik * self.ph_q).real
            return self.fft((self.uq * self.phix + self.vq * self.phiy))
        if self.model == "ybj":
            # niwqg/YBJModel.py:123-133 (no [0,0] zeroing)
            return self.fft((self.u * self.phix + self.v * self.phiy))
        # niwqg/Kernel.py:457-469
        jach = self.fft((self.u * self.phix + self.v * self.phiy))
        jach[0, 0] = 0
        return jach

    # ------------------------------------------------------ budgets / energies
    def spec_var(self, ph):
        """niwqg/Kernel.py:654-658."""
        var_dens = np.abs(ph) ** 2 / self.M ** 2
        var_dens[0, 0] = 0.
        return var_dens.sum()

    def ke_qg(self):
        return 0.5 * self.spec_var(self.wv * self.ph)            # Kernel.py:600-602

    def ke_niw(self):
        return 0.5 * (np.abs(self.phi) ** 2).mean()              # Kernel.py:604-606

    def pe_niw(self):
        """niwqg/Kernel.py:608-611 - side effect: refreshes phix, phiy (F6)."""
        self.phix, self.phiy = self.ifft(self.ik * self.phih), self.ifft(self.il * self.phih)
        return 0.25 * (np.abs(self.phix) ** 2 + np.abs(self.phiy) ** 2).mean() / self.kappa2

    def conc(self):
        """niwqg/Kernel.py:613-619."""
        self.upsilon = np.abs(self.phi) ** 2 - (np.abs(self.phi) ** 2).mean()
        return (self.upsilon * self.q_psi).mean() / self.upsilon.std() / self.q_psi.std()

    def skewness(self):
        return ((self.q_psi ** 3).mean() / (((self.q_psi ** 2).mean()) ** 1.5))   # Kernel.py:621-623

    def ep_phi(self):
        """niwqg/Kernel.py:629-633."""
        return -self.nu4w * (np.abs(self.lapphi) ** 2).mean() \
            - self.nuw * (np.abs(self.phix) ** 2 + np.abs(self.phiy) ** 2).mean() \
            - self.muw * (np.abs(self.phi) ** 2).mean()

    def ep_psi(self):
        """niwqg/Kernel.py:635-640."""
        lap2psi = self.ifft(self.wv4 * self.ph).real
        lapq = self.ifft(-self.wv2 * self.qh).real
        return self.nu4 * (self.q * lap2psi).mean() - self.nu * (self.p * lapq).mean() \
            + self.mu * (self.p * self.q).mean()

    def chi_q(self):
        return -self.nu4 * self.spec_var(self.wv2 * self.qh)     # Kernel.py:642-644

    def chi_phi(self):
        """niwqg/Kernel.py:646-652."""
        lphix, lphiy = self.ifft(-self.ik * self.wv2 * self.phih), \
            self.ifft(-self.il * self.wv2 * self.phih)
        return -0.5 * self.nu4w * (np.abs(lphix) ** 2 + np.abs(lphiy) ** 2).mean() / self.kappa2 \
            - 0.5 * self.nuw * (np.abs(self.lapphi) ** 2).mean() / self.kappa2 \
            - 0.5 * self.muw * (np.abs(self.phix) ** 2 + np.abs(self.phiy) ** 2).mean() / self.kappa2

    def cfl(self):
        """niwqg/Kernel.py:660-662."""
        return np.abs(np.hstack([self.u, self.v, np.abs(self.phi)])).max() * self.dt / self.dx

    def energy_conversion(self):
        """niwqg/Kernel.py:664-701."""
        self.u, self.v = self.ifft(-self.il * self.ph).real, self.ifft(self.ik * self.ph).real
        self._rel_vorticity()
        J_psi_phi = self.u * self.phix + self.v * self.phiy
        self.lapphi = np.fft.ifft2(-self.wv2 * self.phih)
        lap2phi = self.ifft(self.wv4 * self.phih)
        diss_phi = -self.nu4w * lap2phi + self.nuw * self.lapphi - self.muw * self.phi
        J_diss_phi = -(diss_phi * np.conj(J_psi_phi)).imag
        L_diss_phi = 0.5 * (diss_phi * np.conj(self.phi)).real * self.q_psi
        divFw = 0.5 * self.hslash * (np.conj(self.phi) * self.lapphi).imag
        self.gamma1 = (0.5 * self.q_psi * divFw).mean() / self.f
        self.gamma2 = 0.5 * self.hslash * ((np.conj(self.lapphi) * J_psi_phi).real).mean() / self.f
        self.xi1 = J_diss_phi.mean() / self.f
        self.xi2 = L_diss_phi.mean() / self.f
        self.pi = (0.5 * self.phi.mean() * (self.q_psi * np.conj(self.phi)).mean()).imag

    def ke_qg_decomp(self):
        """niwqg/CoupledModel.py:99-113."""
        self.phq = -self.wv2i * self.qh
        self.ke_qg_q = 0.5 * self.spec_var(self.wv * self.phq)
        self.phw = self.wv2i * self.qwh
        self.ke_qg_w = 0.5 * self.spec_var(self.wv * self.phw)
        self.uq, self.vq = self.ifft(-self.il * self.phq).real, self.ifft(self.ik * self.phq).real
        self.uw, self.vw = self.ifft(-self.il * self.phw).real, self.ifft(self.ik * self.phw).real
        self.ke_qg_qw = (self.uq * self.uw).mean() + (self.vq * self.vw).mean()

    # ---------------------------------------------------------------- stepping
    def _budget_rates(self):
        """One stage's (k, p, a) budget tendencies: niwqg/Kernel.py:319-322."""
        self.energy_conversion()
        ks = -(self.gamma1 + self.gamma2) + (self.xi1 + self.xi2) + self.ep_psi()
        ps = self.gamma1 + self.gamma2 + self.chi_phi()
        a_s = self.ep_phi()
        return ks, ps, a_s

    def _refresh(self):
        """niwqg/Kernel.py:337-339."""
        self.phi = self.ifft(self.phih)
        self._invert()
        self._rel_vorticity()

    def _wave_rhs(self):
        """niwqg/Kernel.py:332."""
        return -self.jacobian_psi_phi() - 0.5j * self.fft(self.phi * self.q_psi)

    def step(self):
        if self.model == "ybj":
            return self._step_ybj()
        # niwqg/Kernel.py:307-397
        k1, p1, a1 = self._budget_rates()
        self.qh0 = self.qh.copy()
        Fn0 = -self.jacobian_psi_q()
        self.qh = (self.expch_h * self.qh0 + Fn0 * self.Qh) * self.filtr
        self.qh1 = self.qh.copy()
        self.phih0 = self.phih.copy()
        Fn0w = self._wave_rhs()
        self.phih = (self.expch_hw * self.phih0 + Fn0w * self.Qhw) * self.filtr
        self.phih1 = self.phih.copy()
        self._refresh()

        k2, p2, a2 = self._budget_rates()
        Fna = -self.jacobian_psi_q()
        self.qh = (self.expch_h * self.qh0 + Fna * self.Qh) * self.filtr
        Fnaw = self._wave_rhs()
        self.phih = (self.expch_hw * self.phih0 + Fnaw * self.Qhw) * self.filtr
        self._refresh()

        k3, p3, a3 = self._budget_rates()
        Fnb = -self.jacobian_psi_q()
        self.qh = (self.expch_h * self.qh1 + (2. * Fnb - Fn0) * self.Qh) * self.filtr
        Fnbw = self._wave_rhs()
        self.phih = (self.expch_hw * self.phih1 + (2. * Fnbw - Fn0w) * self.Qhw) * self.filtr
        self._refresh()

        k4, p4, a4 = self._budget_rates()
        Fnc = -self.jacobian_psi_q()
        self.qh = (self.expch * self.qh0 + Fn0 * self.f0 + 2. * (Fna + Fnb) * self.fab
                   + Fnc * self.fc) * self.filtr
        Fncw = self._wave_rhs()
        self.phih = (self.expchw * self.phih0 + Fn0w * self.f0w + 2. * (Fnaw + Fnbw) * self.fabw
                     + Fncw * self.fcw) * self.filtr

        self.Ke += self.dt * (k1 + 2 * (k2 + k3) + k4) / 6.
        self.Pw += self.dt * (p1 + 2 * (p2 + p3) + p4) / 6.
        self.Kw += self.dt * (a1 + 2 * (a2 + a3) + a4) / 6.
        self._refresh()

    def _grad_phi(self):
        self.phix, self.phiy = self.ifft(self.ik * self.phih), self.ifft(self.il * self.phih)  # YBJModel.py:135-139

    def _step_ybj(self):
        """niwqg/YBJModel.py:52-87 (phi stays stale through the stages, F7)."""
        self.phih0 = self.phih.copy()
        self._grad_phi()
        Fn0w = self._wave_rhs()
        self.phih = (self.expch_hw * self.phih0 + Fn0w * self.Qhw) * self.filtr
        self.phih1 = self.phih.copy()
        self._grad_phi()
        Fnaw = self._wave_rhs()
        self.phih = (self.expch_hw * self.phih0 + Fnaw * self.Qhw) * self.filtr
        self._grad_phi()
        Fnbw = self._wave_rhs()
        self.phih = (self.expch_hw * self.phih1 + (2. * Fnbw - Fn0w) * self.Qhw) * self.filtr
        self._rel_vorticity()
        self._grad_phi()
        Fncw = self._wave_rhs()
        self.phih = (self.expchw * self.phih0 + Fn0w * self.f0w + 2. * (Fnaw + Fnbw) * self.fabw
                     + Fncw * self.fcw) * self.filtr
        self.phi = self.ifft(self.phih)

    # ----------------------------------------------------- diagnostics / driver
    DIAG_ORDER = ("time", "Ke", "Pw", "Kw", "ke_qg", "ens", "ke_niw", "cke_niw", "ike_niw",
                  "pe_niw", "conc_niw", "skew", "gamma_r", "gamma_a", "xi_r", "xi_a", "pi",
                  "ep_phi", "ep_psi", "chi_q", "chi_phi")

    def tick(self):
        """niwqg/Diagnostics.py:41-58 with the registry of Kernel.py:718-868 and
        CoupledModel.py:115-143, evaluated in registration order (pe_niw's
        phix/phiy refresh happens before ep_phi/chi_phi read them)."""
        if self.tc % self.tdiags:
            return
        self.energy_conversion()                           # Kernel.py:875-878
        self.ke_niw_d = self.ke_niw()                       # Kernel.py:703-706
        self.cke_niw = 0.5 * (np.abs(self.phi.mean()) ** 2)
        self.ike_niw = self.ke_niw_d - self.cke_niw
        if self.model in ("coupled", "ql"):
            self.ke_qg_decomp()
        rec = {}
        rec["time"] = self.t
        rec["Ke"], rec["Pw"], rec["Kw"] = self.Ke, self.Pw, self.Kw
        rec["ke_qg"] = self.ke_qg()
        rec["ens"] = 0.5 * (self.q ** 2).mean()
        rec["ke_niw"], rec["cke_niw"], rec["ike_niw"] = self.ke_niw_d, self.cke_niw, self.ike_niw
        rec["pe_niw"] = self.pe_niw()
        rec["conc_niw"] = self.conc()
        rec["skew"] = self.skewness()
        rec["gamma_r"], rec["gamma_a"] = self.gamma1, self.gamma2
        rec["xi_r"], rec["xi_a"], rec["pi"] = self.xi1, self.xi2, self.pi
        rec["ep_phi"] = self.ep_phi()
        rec["ep_psi"] = self.ep_psi()
        rec["chi_q"] = self.chi_q()
        rec["chi_phi"] = self.chi_phi()
        if self.model in ("coupled", "ql"):
            rec["ke_qg_q"], rec["ke_qg_w"], rec["ke_qg_qw"] = self.ke_qg_q, self.ke_qg_w, self.ke_qg_qw
        for name, val in rec.items():
            self.diag.setdefault(name, []).append(val)

    def status(self):
        """niwqg/Kernel.py:587-598 (clock advance + status/CFL every twrite steps)."""
        self.tc += 1
        self.t += self.dt
        if (self.tc % self.twrite) == 0:
            self.ke = self.ke_qg()
            self.kew = self.ke_niw()
            self.pew = self.pe_niw()
            self.cfl_now = self.cfl()
            assert self.cfl_now < self.cflmax, "CFL condition violated"

    def step_forward(self):
        """niwqg/Kernel.py:205-217 without the disk writes."""
        self.step()
        self.tick()
        self.status()

    def run(self):
        while self.t < self.tmax:                          # Kernel.py:198-199
            self.step_forward()

    def diagnostics(self):
        return {k: np.array(v) for k, v in self.diag.items()}


class QGOracle(object):
    """Stand-alone QG model oracle (rfft2/irfft2, half spectrum).

    Follows niwqg/QGModel.py; constructor keywords/defaults :65-91.  The
    passive-scalar branch (:345-394) is included (SURVEY.md section 8f N4).
    """

    def __init__(self, nx=128, ny=None, L=5e5, dt=10000., twrite=1000, tmax=250000.,
                 use_filter=True, U=.0, nu4=5.e9, nu=0, mu=0, beta=0, passive_scalar=False,
                 nu4c=5.e9, nuc=0, muc=0, dealias=False, tdiags=10):
        self.nx, self.ny, self.L, self.W = nx, nx, L, L
        self.dt, self.twrite, self.tmax, self.tdiags = dt, twrite, tmax, tdiags
        self.passive_scalar, self.dealias, self.use_filter = passive_scalar, dealias, use_filter
        self.U, self.beta, self.nu4, self.nu, self.mu = U, beta, nu4, nu, mu
        self.nu4c, self.nuc, self.muc = nu4c, nuc, muc
        # grid: QGModel.py:232-269
        self.x, self.y = np.meshgrid(np.arange(0.5, nx, 1.) / nx * L, np.arange(0.5, nx, 1.) / nx * L)
        self.dk = self.dl = 2. * np.pi / L
        self.nl, self.nk = nx, nx // 2 + 1
        self.ll = self.dl * np.append(np.arange(0., nx / 2), np.arange(-nx / 2, 0.))
        self.kk = self.dk * np.arange(0., self.nk)
        self.k, self.l = np.meshgrid(self.kk, self.ll)
        self.ik, self.il = 1j * self.k, 1j * self.l
        self.dx = self.dy = L / nx
        self.M = nx * nx
        self.wv2 = self.k ** 2 + self.l ** 2
        self.wv = np.sqrt(self.wv2)
        self.wv4 = self.wv2 ** 2
        nz = self.wv2 != 0.
        self.wv2i = np.zeros_like(self.wv2)
        self.wv2i[nz] = self.wv2[nz] ** -1
        # variables: QGModel.py:141-158
        self.q = np.zeros((nx, nx))
        self.qh = np.zeros((nx, self.nk), np.complex128)
        self.p = np.zeros((nx, nx))
        self.ph = np.zeros((nx, self.nk), np.complex128)
        # filter: QGModel.py:283-301 (the dealias branch of the reference raises
        # TypeError from float slices - SURVEY.md section 8c defect 2 - integer slices here)
        self.filtr = spectral_filter(self.k, self.l, self.dx, self.dy, use_filter, dealias, nx, nx)
        # coefficients: QGModel.py:410-466
        c = np.zeros((self.nl, self.nk), np.complex128)
        c += -self.nu4 * self.wv4 - self.nu * self.wv2 - self.mu - 1j * self.k * self.U
        c += self.beta * self.ik * self.wv2i
        (self.expch, self.expch_h, self.Qh, self.f0, self.fab, self.fc) = etdrk4_tables(c * dt, dt)
        if passive_scalar:
            c = np.zeros((self.nl, self.nk), np.complex128)
            c += -self.nu4c * self.wv4 - self.nuc * self.wv2 - self.muc
            (self.expchc, self.expch_hc, self.Qhc, self.f0c, self.fabc, self.fcc) = \
                etdrk4_tables(c * dt, dt)
        self.t = 0
        self.tc = 0
        self.cflmax = .5
        self.fft = lambda x: np.fft.rfft2(x)               # QGModel.py:551-552
        self.ifft = lambda x: np.fft.irfft2(x)
        self.diag = {}

    def spec_var(self, ph):
        """niwqg/QGModel.py:611-619."""
        var_dens = 2. * np.abs(ph) ** 2 / self.M ** 2
        var_dens[:, 0] *= 0.5
        var_dens[:, -1] *= 0.5
        var_dens[0, 0] = 0
        return var_dens.sum()

    def _invert(self):
        self.ph = -self.wv2i * (self.qh)                    # QGModel.py:497-505
        self.p = self.ifft(self.ph)

    def set_q(self, q):
        self.q = q                                          # QGModel.py:507-520
        self.qh = self.fft(self.q)
        self._invert()
        self.Ke = self.ke_qg()

    def set_c(self, c):
        self.c = c                                          # QGModel.py:522-534
        self.ch = self.fft(self.c)
        self.cvar = self.spec_var(self.ch)

    def ke_qg(self):
        return 0.5 * self.spec_var(self.wv * self.ph)       # QGModel.py:577-579

    def ep_psi(self):
        lap2psi = self.ifft(self.wv4 * self.ph)             # QGModel.py:588-593
        lapq = self.ifft(-self.wv2 * self.qh)
        return self.nu4 * (self.q * lap2psi).mean() - self.nu * (self.p * lapq).mean() \
            + self.mu * (self.p * self.q).mean()

    def ep_c(self):
        return -2 * self.nu4c * (self.lapc ** 2).mean() - 2 * self.nu * self.gradC2 \
            - 2 * self.muc * self.C2                        # QGModel.py:595-598

    def chi_c(self):
        lap2c = self.ifft(self.wv4 * self.ch)               # QGModel.py:600-604
        return 2 * self.nu4c * (lap2c * self.lapc).mean() - 2 * self.nu * (self.lapc ** 2).mean() \
            - 2 * self.muc * self.gradC2

    def chi_q(self):
        return -self.nu4 * self.spec_var(self.wv2 * self.qh)   # QGModel.py:606-609

    def cfl(self):
        self.u = self.ifft(-self.il * self.ph)              # QGModel.py:621-629
        self.v = self.ifft(self.ik * self.ph)
        return np.abs(np.hstack([self.u, self.v])).max() * self.dt / self.dx

    def jacobian_psi_q(self):
        """niwqg/QGModel.py:469-481."""
        self.u, self.v = self.ifft(-self.il * self.ph).real, self.ifft(self.ik * self.ph).real
        q = self.ifft(self.qh).real
        return self.ik * self.fft(self.u * q) + self.il * self.fft(self.v * q)

    def jacobian_psi_c(self):
        self.c = self.ifft(self.ch).real                    # QGModel.py:483-495
        return self.ik * self.fft(self.u * self.c) + self.il * self.fft(self.v * self.c)

    def derived_fields(self):
        """niwqg/QGModel.py:724-737."""
        if self.passive_scalar:
            self.C2 = self.spec_var(self.ch)
            self.gradC2 = self.spec_var(self.wv * self.ch)
            self.lapc = self.ifft(-self.wv2 * self.ch)
            self.Gamma_c = 2 * (self.lapc * self.ifft(self.jacobian_psi_c())).mean()
        else:
            self.C2, self.gradC2, self.cvar = 0., 0., 0.
            self.c, self.ch = 0., 0.
            self.lapc, self.Gamma_c = np.array([0.]), 0.

    def step(self):
        """niwqg/QGModel.py:328-407."""
        ps = self.passive_scalar
        self.qh0 = self.qh.copy()
        Fn0 = -self.jacobian_psi_q()
        self.qh = (self.expch_h * self.qh0 + Fn0 * self.Qh) * self.filtr
        self.qh1 = self.qh.copy()
        if ps:
            self.ch0 = self.ch.copy()
            Fn0c = -self.jacobian_psi_c()
            self.ch = (self.expch_hc * self.ch0 + Fn0c * self.Qhc) * self.filtr
            self.ch1 = self.ch.copy()
            self.derived_fields()
            c1 = self.ep_c()
        self._invert()
        k1 = self.ep_psi()

        Fna = -self.jacobian_psi_q()
        self.qh = (self.expch_h * self.qh0 + Fna * self.Qh) * self.filtr
        if ps:
            Fnac = -self.jacobian_psi_c()
            self.ch = (self.expch_hc * self.ch0 + Fnac * self.Qhc) * self.filtr
            self.derived_fields()
            c2 = self.ep_c()
        self._invert()
        k2 = self.ep_psi()

        Fnb = -self.jacobian_psi_q()
        self.qh = (self.expch_h * self.qh1 + (2. * Fnb - Fn0) * self.Qh) * self.filtr
        if ps:
            Fnbc = -self.jacobian_psi_c()
            self.ch = (self.expch_hc * self.ch1 + (2. * Fnbc - Fn0c) * self.Qhc) * self.filtr
            self.derived_fields()
            c3 = self.ep_c()
        self._invert()
        k3 = self.ep_psi()

        Fnc = -self.jacobian_psi_q()
        self.qh = (self.expch * self.qh0 + Fn0 * self.f0 + 2. * (Fna + Fnb) * self.fab
                   + Fnc * self.fc) * self.filtr
        if ps:
            Fncc = -self.jacobian_psi_c()
            self.ch = (self.expchc * self.ch0 + Fn0c * self.f0c + 2. * (Fnac + Fnbc) * self.fabc
                       + Fncc * self.fcc) * self.filtr
            self.derived_fields()
            c4 = self.ep_c()
            self.cvar += self.dt * (c1 + 2 * (c2 + c3) + c4) / 6.
        self._invert()
        self.q = self.ifft(self.qh).real
        if ps:
            self.c = self.ifft(self.ch).real
        k4 = self.ep_psi()
        self.Ke += self.dt * (k1 + 2 * (k2 + k3) + k4) / 6.

    def tick(self):
        """niwqg/Diagnostics.py:41-58 with the registry of QGModel.py:632-722."""
        if self.tc % self.tdiags:
            return
        self.derived_fields()
        rec = {"time": self.t, "ke_qg": self.ke_qg(), "Ke": self.Ke,
               "ens": 0.5 * (self.q ** 2).mean(), "ep_psi": self.ep_psi(), "chi_q": self.chi_q(),
               "C2": self.C2, "cvar": self.cvar, "gradC2": self.gradC2, "Gamma_c": self.Gamma_c}
        rec["ep_c"] = self.ep_c()
        rec["chi_c"] = self.chi_c()
        for name, val in rec.items():
            self.diag.setdefault(name, []).append(val)

    def status(self):
        self.tc += 1                                        # QGModel.py:571-582
        self.t += self.dt
        if (self.tc % self.twrite) == 0:
            self.ke = self.ke_qg()
            self.cfl_now = self.cfl()
            assert self.cfl_now < self.cflmax, "CFL condition violated"

    def step_forward(self):
        self.step()
        self.tick()
        self.status()

    def run(self):
        while self.t < self.tmax:
            self.step_forward()

    def diagnostics(self):
        return {k: np.array(v) for k, v in self.diag.items()}


# ----------------------------------------------------------------------------
# Initial conditions (restated so the oracle is self-contained on the GPU box).
# ----------------------------------------------------------------------------
def lamb_dipole(model, U=.01, R=1.):
    """niwqg/InitialConditions.py:77-114 (vectorised: the reference's Python
    double loop only guards the r==0 division)."""
    from scipy import special
    N = model.nx
    x, y = model.x, model.y
    x0, y0 = x[N // 2, N // 2], y[N // 2, N // 2]
    r = np.sqrt((x - x0) ** 2 + (y - y0) ** 2)
    s = np.zeros_like(r)
    nz = r != 0.
    s[nz] = (y[nz] - y0) / r[nz]
    lam = (3.8317) / R
    C = -(2. * U * lam) / (special.j0(lam * R))
    q = np.zeros_like(r)
    q[r <= R] = C * special.j1(lam * r[r <= R]) * s[r <= R]
    return q


def mcwilliams1984(model, k0=6, E=0.5):
    """niwqg/InitialConditions.py:4-41 (consumes the global numpy RNG)."""
    ckappa = np.zeros_like(model.wv2)
    nhx, nhy = model.wv2.shape
    kc2 = k0 ** 2
    fk = model.wv != 0
    ckappa[fk] = np.sqrt(model.wv2[fk] * (1. + (model.wv2[fk] / kc2) ** 2)) ** -1
    phase = np.random.rand(nhx, nhy) * 2 * np.pi
    ph = ckappa * np.cos(phase) + 1j * ckappa * np.sin(phase)
    ph = model.fft(model.ifft(ph).real)
    Eaux = 0.5 * model.spec_var(model.wv * ph)
    pih = np.sqrt(E / Eaux) * ph
    qih = -model.wv2 * pih
    return model.ifft(qih).real
