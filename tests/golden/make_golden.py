"""Generate golden vectors from the UNMODIFIED reference (a checkout of the niwqg project; the
directory that holds its ``niwqg`` package):

    python tests/golden/make_golden.py REFERENCE_DIR [CASE ...]

The reference imports ``h5py`` at module top (niwqg/Kernel.py:4) but only
dereferences it when save_to_disk=True; h5py is not installed here, so a stub
module is placed on sys.modules first.  Nothing from the reference is copied:
it is imported, run through its public API, and its outputs are stored.
"""
import os, sys, types
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def import_reference(ref_dir):
    if "h5py" not in sys.modules:
        try:
            import h5py  # noqa: F401
        except Exception:
            sys.modules["h5py"] = types.ModuleType("h5py")
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    import logging
    import niwqg
    from niwqg import CoupledModel, UnCoupledModel, YBJModel, QGModel, InitialConditions
    logging.getLogger("niwqg.Kernel").setLevel(100)
    logging.getLogger("niwqg.QGModel").setLevel(100)
    logging.disable(logging.CRITICAL)

    class RepairedQL(CoupledModel.Model):
        """SURVEY.md section 8c: QLModel.py does not run (F8); the QL oracle is
        CoupledModel with the wave advection body of niwqg/QLModel.py:65-67."""
        def jacobian_psi_phi(self):
            self.ph_q = -self.wv2i * self.qh
            self.uq, self.vq = self.ifft(-self.il * self.ph_q).real, self.ifft(self.ik * self.ph_q).real
            return self.fft((self.uq * self.phix + self.vq * self.phiy))

    ctor = {"coupled": CoupledModel.Model, "uncoupled": UnCoupledModel.Model,
            "ybj": YBJModel.Model, "ql": RepairedQL, "qg": QGModel.Model}
    return ctor, InitialConditions


def lamb_params(nx, use_filter, tdiags, nsteps, qg=False):
    """Parameters of examples/LambDipole.py:22-52 / LambDipole_qg.py:21-45 scaled to nx."""
    L = 2 * np.pi * 200e3
    k0 = 10 * (2 * np.pi / L)
    U0 = 1.e-1
    Te = (U0 * k0) ** -1
    if qg:
        dt = .05 * Te * 128 / nx
        kw = dict(L=L, nx=nx, dt=dt, tmax=nsteps * dt - 0.5 * dt, twrite=7, nu4=7.5e8 * (128 / nx) ** 4,
                  use_filter=use_filter, U=-U0, tdiags=tdiags, beta=0.)
    else:
        dt = .025 * Te * 128 / nx
        kw = dict(L=L, nx=nx, dt=dt, tmax=nsteps * dt - 0.5 * dt, twrite=7, m=2 * np.pi / 280, N=0.01,
                  f=1.e-4, nu4=5e11 * (128 / nx) ** 4, nu4w=0., nu=20, nuw=50., mu=0., muw=0.,
                  use_filter=use_filter, U=-U0, tdiags=tdiags)
    return kw, U0, k0


CASES = [
    # name, model, nx, use_filter, tdiags, nsteps, ic
    ("coupled_lamb64_filt", "coupled", 64, True, 2, 10, "lamb"),
    ("coupled_lamb64_nofilt", "coupled", 64, False, 2, 10, "lamb"),
    ("uncoupled_lamb64_filt", "uncoupled", 64, True, 3, 10, "lamb"),
    ("uncoupled_lamb64_nofilt", "uncoupled", 64, False, 3, 10, "lamb"),
    ("ql_lamb64_filt", "ql", 64, True, 2, 10, "lamb"),
    ("ql_lamb64_nofilt", "ql", 64, False, 2, 10, "lamb"),
    ("ybj_lamb64_filt", "ybj", 64, True, 2, 10, "lamb"),
    ("ybj_lamb64_nofilt", "ybj", 64, False, 2, 10, "lamb"),
    ("coupled_rand64_filt", "coupled", 64, True, 5, 10, "mcw"),
    ("ybj_rand64_filt", "ybj", 64, True, 5, 10, "mcw"),
    ("coupled_lamb128_nofilt_100", "coupled", 128, False, 1, 100, "lamb"),
    ("coupled_lamb128_filt_100", "coupled", 128, True, 10, 100, "lamb"),
    ("qg_lamb64_filt", "qg", 64, True, 2, 20, "lamb"),
    ("qg_lamb128_nofilt_100", "qg", 128, False, 1, 100, "lamb"),
    ("qg_scalar64_nofilt", "qgc", 64, False, 1, 20, "lamb"),
    # parameter branches (keywords in tests/cases.py:EXTRA)
    ("coupled_lamb64_diss", "coupled", 64, True, 1, 10, "lamb"),
    ("coupled_lamb64_dealias", "coupled", 64, False, 2, 10, "lamb"),
    ("uncoupled_lamb64_diss", "uncoupled", 64, True, 2, 10, "lamb"),
    ("ql_lamb64_diss", "ql", 64, True, 2, 10, "lamb"),
    ("qg_lamb64_beta", "qg", 64, True, 2, 20, "lamb"),
]


def run_case(ctor, ic, name, model, nx, use_filter, tdiags, nsteps, icname):
    qg = model in ("qg", "qgc")
    kw, U0, k0 = lamb_params(nx, use_filter, tdiags, nsteps, qg=qg)
    if model == "qgc":
        kw.update(passive_scalar=True, nu4c=3.e9 * (128 / nx) ** 4, nuc=0)
    sys.path.insert(0, os.path.dirname(HERE))
    from cases import EXTRA
    kw.update(EXTRA.get(name, {}))
    m = ctor["qg" if qg else model](**kw)
    if icname == "lamb":
        q = ic.LambDipole(m, U=U0, R=2 * np.pi / k0)
    else:
        np.random.seed(7)
        q = ic.McWilliams1984(m, k0=k0, E=U0 ** 2 / 2)
    out = {}
    if nx <= 64:
        out["q0"] = q.copy()
    m.set_q(q)
    if model == "qgc":
        c = ic.PlaneWave(m, k=k0 / 5, l=k0 / 5).real
        out["c0"] = c.copy()
        m.set_c(c)
    if not qg:
        phi = (np.ones_like(q) + 1j) * (2 * U0) / np.sqrt(2)
        m.set_phi(phi)
    # first step recorded separately (F5 state-seeding semantics show up here)
    m._step_forward()
    out["q_1"] = np.array(m.q)
    if not qg:
        out["phi_1"] = np.array(m.phi)
    while m.t < m.tmax:
        m._step_forward()
    assert m.tc == nsteps, (m.tc, nsteps)
    out["q"] = np.array(m.q)
    out["Ke"] = np.float64(m.Ke)
    if not qg:
        out["phi"] = np.array(m.phi)
        out["Pw"] = np.float64(m.Pw)
        out["Kw"] = np.float64(m.Kw)
    if model == "qgc":
        out["c"] = np.array(m.c)
        out["cvar"] = np.float64(m.cvar)
    for dn, d in m.diagnostics.items():
        if "value" in d:
            out["diag_" + dn] = np.atleast_1d(np.array(d["value"], dtype=np.float64))
    out["nsteps"] = np.int64(nsteps)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "ok", {k: getattr(v, "shape", None) for k, v in out.items() if not k.startswith("diag_")})


def coefficient_case(ctor):
    """ETDRK4 tables + filter of a small Coupled model (pins Kernel.py:400-454, :267-284)."""
    kw, U0, k0 = lamb_params(32, True, 1, 1)
    m = ctor["coupled"](**kw)
    names = ["expch", "expch_h", "Qh", "f0", "fab", "fc", "expchw", "expch_hw", "Qhw", "f0w", "fabw", "fcw", "filtr"]
    np.savez_compressed(os.path.join(HERE, "coeffs_coupled32.npz"), **{n: getattr(m, n) for n in names})
    print("coeffs ok")


def reference_tests_known_answers(ctor):
    """The reference's own assertions for this path (niwqg/tests/*.py), evaluated on
    the reference; stored so the same assertions can be replayed on the CUDA path."""
    rng = np.random.RandomState(11)
    m = ctor["coupled"](use_filter=False)
    qi = rng.randn(m.ny, m.nx)
    phii = rng.randn(m.ny, m.nx) + 1j * rng.randn(m.ny, m.nx)
    out = {"qi": qi, "phii": phii, "fft_qi": m.fft(qi), "fft_phii": m.fft(phii)}
    m.set_q(qi); m.set_phi(phii)
    out["spec_var_q"] = np.float64(m.spec_var(m.qh)); out["spec_var_phi"] = np.float64(m.spec_var(m.phih))
    np.savez_compressed(os.path.join(HERE, "reftests_fft128.npz"), **out)
    print("reftests ok")


if __name__ == "__main__":
    if len(sys.argv) < 2:
        raise SystemExit(__doc__)
    ctor, ic = import_reference(os.path.abspath(sys.argv[1]))
    only = sys.argv[2:]          # optional: regenerate just these cases
    for case in CASES:
        if not only or case[0] in only:
            run_case(ctor, ic, *case)
    if not only:
        coefficient_case(ctor)
        reference_tests_known_answers(ctor)
