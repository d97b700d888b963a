"""Shared case builders for the parity tests: same parameters/ICs as tests/golden/make_golden.py."""
import os
import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

CASES = {
    # name: (model, nx, use_filter, tdiags, nsteps, ic)
    "coupled_lamb64_filt": ("coupled", 64, True, 2, 10, "lamb"),
    "coupled_lamb64_nofilt": ("coupled", 64, False, 2, 10, "lamb"),
    "uncoupled_lamb64_filt": ("uncoupled", 64, True, 3, 10, "lamb"),
    "uncoupled_lamb64_nofilt": ("uncoupled", 64, False, 3, 10, "lamb"),
    "ql_lamb64_filt": ("ql", 64, True, 2, 10, "lamb"),
    "ql_lamb64_nofilt": ("ql", 64, False, 2, 10, "lamb"),
    "ybj_lamb64_filt": ("ybj", 64, True, 2, 10, "lamb"),
    "ybj_lamb64_nofilt": ("ybj", 64, False, 2, 10, "lamb"),
    "coupled_rand64_filt": ("coupled", 64, True, 5, 10, "mcw"),
    "ybj_rand64_filt": ("ybj", 64, True, 5, 10, "mcw"),
    "coupled_lamb128_nofilt_100": ("coupled", 128, False, 1, 100, "lamb"),
    "coupled_lamb128_filt_100": ("coupled", 128, True, 10, 100, "lamb"),
    "qg_lamb64_filt": ("qg", 64, True, 2, 20, "lamb"),
    "qg_lamb128_nofilt_100": ("qg", 128, False, 1, 100, "lamb"),
    "qg_scalar64_nofilt": ("qgc", 64, False, 1, 20, "lamb"),
    # parameter branches no other case touches (constructor keywords in EXTRA below)
    "coupled_lamb64_diss": ("coupled", 64, True, 1, 10, "lamb"),       # nu4w, mu, muw != 0 (Kernel.py:688-689, :646-652)
    "coupled_lamb64_dealias": ("coupled", 64, False, 2, 10, "lamb"),   # 2/3-rule mask (Kernel.py:277-281)
    "uncoupled_lamb64_diss": ("uncoupled", 64, True, 2, 10, "lamb"),   # nu4w != 0 without the wave PV
    "ql_lamb64_diss": ("ql", 64, True, 2, 10, "lamb"),                 # nu4w != 0 on the physical-space budget path
    "qg_lamb64_beta": ("qg", 64, True, 2, 20, "lamb"),                 # beta != 0 (QGModel.py:428)
}

EXTRA = {
    "coupled_lamb64_diss": dict(nu4w=2.e11, mu=2.e-8, muw=3.e-8),
    "coupled_lamb64_dealias": dict(dealias=True),
    "uncoupled_lamb64_diss": dict(nu4w=2.e11, muw=3.e-8),
    "ql_lamb64_diss": dict(nu4w=2.e11, mu=2.e-8, muw=3.e-8),
    "qg_lamb64_beta": dict(beta=2.e-11, mu=1.e-8),
}


def lamb_params(nx, use_filter, tdiags, nsteps, qg=False):
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


def case_params(name, **over):
    """(model kind, constructor keywords, U0, k0) of a golden case, as tests/golden/make_golden.py sets it up."""
    model, nx, use_filter, tdiags, nsteps, icname = CASES[name]
    qg = model in ("qg", "qgc")
    kw, U0, k0 = lamb_params(nx, use_filter, tdiags, nsteps, qg=qg)
    if model == "qgc":
        kw.update(passive_scalar=True, nu4c=3.e9 * (128 / nx) ** 4, nuc=0)
    kw.update(EXTRA.get(name, {}))
    kw.update(over)
    return model, kw, U0, k0


def case_ics(name, grid, U0, k0):
    """Initial fields of a golden case on the grid of ``grid`` (anything with nx, x, y): {"q", "phi" or "c"}."""
    from oracle import niwqg_oracle as orc
    model, icname = CASES[name][0], CASES[name][5]
    if icname == "lamb":
        q = orc.lamb_dipole(grid, U=U0, R=2 * np.pi / k0)
    else:
        # the random IC needs the reference FFT arithmetic to be bit-identical: take it from the golden file
        q = load_golden(name)["q0"]
    ics = {"q": q}
    if model == "qgc":
        ics["c"] = np.exp(1j * (k0 / 5 * grid.x + k0 / 5 * grid.y) + 0.).real
    elif model != "qg":
        ics["phi"] = (np.ones_like(q) + 1j) * (2 * U0) / np.sqrt(2)
    return ics


def plane_wave_factor(kx, ky, N, L, t, nu4=0., beta=0., U=0.):
    """exp(c t) of the linear operator c = -nu4 |K|^4 - i k U + i beta k / |K|^2 at the mode (kx, ky) (indices, ky
    signed by the FFT convention).  A single plane wave has J(psi, q) = 0, so its coefficient evolves by exactly this
    factor: a hyperviscously decaying, Doppler-shifted Rossby wave (QGModel.py:410-466 without nu and mu)."""
    k = 2 * np.pi / L * kx
    l = 2 * np.pi / L * (ky if ky < N // 2 else ky - N)
    wv2 = k * k + l * l
    return np.exp((-nu4 * wv2 * wv2 - 1j * k * U + 1j * beta * k / wv2) * t)


def plane_wave_coefficient(kx, ky, N, L, A=1.):
    """Spectral coefficient at (ky, kx) of A sin(k x + l y) sampled at the cell centres x = (i + 1/2) L / N."""
    dx = L / N
    k, l = 2 * np.pi / L * kx, 2 * np.pi / L * ky
    return A * N * N / 2j * np.exp(0.5j * (k + l) * dx)


# Every diagnostic is compared against the magnitude of the budget it belongs to: cross terms and
# tendencies are differences of much larger numbers, so "relative to itself" is not meaningful for them.
QG_ENERGY = ("Ke", "ke_qg", "ke_qg_q", "ke_qg_w", "ke_qg_qw")
WAVE_ENERGY = ("Kw", "ke_niw", "cke_niw", "ike_niw", "Pw", "pe_niw")
TENDENCIES = ("gamma_r", "gamma_a", "xi_r", "xi_a", "pi", "ep_phi", "ep_psi", "chi_phi")
SCALAR_TEND = ("ep_c", "chi_c", "Gamma_c")
TOL_DIAG = 1e-9


def diag_scale(dn, ref, g):
    """Scale of diagnostic ``dn`` (reference series ``ref``); ``g`` maps "diag_<name>" to the reference series."""
    def mx(names):
        return max([float(np.max(np.abs(g["diag_" + n]))) for n in names if "diag_" + n in g] + [0.0])
    if dn in ("skew", "conc_niw"):
        return 1.0                                   # normalised O(1) quantities
    if dn in QG_ENERGY:
        return mx(("ke_qg",))
    if dn in WAVE_ENERGY:
        # Pw is compared on its own scale once it has grown; early on it is rounding noise of Kw
        return max(float(np.max(np.abs(ref))), 1e-6 * mx(("ke_niw",)))
    if dn in TENDENCIES:
        return mx(TENDENCIES)
    return float(np.max(np.abs(ref)))


def diag_check(dn, got, ref, g, tol=TOL_DIAG):
    ref = np.asarray(ref, float); got = np.asarray(got, float)
    assert got.shape == ref.shape, (dn, got.shape, ref.shape)
    ok = np.isfinite(ref)                            # conc_niw is 0/0 for a uniform wave at t=0 in the reference too
    ref, got = ref[ok], got[ok]
    if ref.size == 0:
        return
    scale = diag_scale(dn, ref, g)
    if scale == 0:
        assert np.max(np.abs(got)) < 1e-20, dn
        return
    err = float(np.max(np.abs(got - ref)) / scale)
    assert err <= tol, (dn, err, got[:3], ref[:3])


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz")))


def rel_l2(a, b):
    a = np.asarray(a); b = np.asarray(b)
    return float(np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-300))
