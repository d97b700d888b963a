"""Pin the CPU oracle (oracle/niwqg_oracle.py) against golden vectors produced by the
unmodified reference (tests/golden/make_golden.py).  Bit-exact: same numpy ops, same order."""
import numpy as np
import pytest

from cases import CASES, EXTRA, lamb_params, load_golden
from oracle import niwqg_oracle as orc


def build_oracle(name):
    model, nx, use_filter, tdiags, nsteps, icname = CASES[name]
    qg = model in ("qg", "qgc")
    kw, U0, k0 = lamb_params(nx, use_filter, tdiags, nsteps, qg=qg)
    if qg:
        if model == "qgc":
            kw.update(passive_scalar=True, nu4c=3.e9 * (128 / nx) ** 4, nuc=0)
        kw.update(EXTRA.get(name, {}))
        m = orc.QGOracle(**kw)
    else:
        kw.update(EXTRA.get(name, {}))
        m = orc.NIWQGOracle(model=model, **kw)
    if icname == "lamb":
        q = orc.lamb_dipole(m, U=U0, R=2 * np.pi / k0)
    else:
        np.random.seed(7)
        q = orc.mcwilliams1984(m, k0=k0, E=U0 ** 2 / 2)
    m.set_q(q)
    if model == "qgc":
        m.set_c(np.exp(1j * (k0 / 5 * m.x + k0 / 5 * m.y) + 0.).real)   # InitialConditions.py:167
    if not qg:
        m.set_phi((np.ones_like(q) + 1j) * (2 * U0) / np.sqrt(2))
    return m, q


SMALL = [n for n in CASES if CASES[n][1] <= 64]


@pytest.mark.parametrize("name", SMALL + ["coupled_lamb128_nofilt_100", "qg_lamb128_nofilt_100"])
def test_oracle_matches_golden_bitwise(name):
    g = load_golden(name)
    m, q0 = build_oracle(name)
    if "q0" in g:
        assert np.array_equal(q0, g["q0"]), "initial condition differs from the reference's"
    m.step_forward()
    assert np.array_equal(m.q, g["q_1"])
    if "phi_1" in g:
        assert np.array_equal(m.phi, g["phi_1"])
    while m.t < m.tmax:
        m.step_forward()
    assert m.tc == int(g["nsteps"])
    assert np.array_equal(m.q, g["q"])
    assert float(m.Ke) == float(g["Ke"])
    if "phi" in g:
        assert np.array_equal(m.phi, g["phi"])
        assert float(m.Pw) == float(g["Pw"]) and float(m.Kw) == float(g["Kw"])
    if "c" in g:
        assert np.array_equal(m.c, g["c"]) and float(m.cvar) == float(g["cvar"])
    d = m.diagnostics()
    for k, v in g.items():
        if k.startswith("diag_"):
            assert np.array_equal(np.atleast_1d(d[k[5:]]).astype(np.float64), v, equal_nan=True), k


def test_oracle_coefficients_match_golden():
    g = load_golden("coeffs_coupled32")
    kw, U0, k0 = lamb_params(32, True, 1, 1)
    m = orc.NIWQGOracle(model="coupled", **kw)
    for n, v in g.items():
        assert np.array_equal(getattr(m, n), v), n


def test_reference_fft_known_answers():
    """niwqg/tests/test_fft.py: round trip + Parseval, on the oracle's transforms."""
    g = load_golden("reftests_fft128")
    m = orc.NIWQGOracle(model="coupled", use_filter=False)
    assert np.array_equal(m.fft(g["qi"]), g["fft_qi"])
    assert np.allclose(m.ifft(m.fft(g["phii"])), g["phii"], rtol=1e-15)
    m.set_q(g["qi"]); m.set_phi(g["phii"])
    assert float(m.spec_var(m.qh)) == float(g["spec_var_q"])
    assert abs(m.spec_var(m.phih) - g["phii"].var()) / g["phii"].var() < 1e-15


def test_plane_wave_formula_matches_qg_oracle():
    """The exact single-mode solution the GPU plane-wave tests use (cases.plane_wave_factor: hyperviscous decay,
    Doppler shift and Rossby phase of the linear operator) against QGOracle stepping the same wave at 64^2."""
    from cases import plane_wave_coefficient, plane_wave_factor
    N, L, dt, nsteps, A = 64, 5e5, 2000., 3, 1e-14
    x = (np.arange(N) + 0.5) / N * L
    for kx, ky in ((5, 29), (29, 3), (17, 17)):
        wv2 = (2 * np.pi / L) ** 2 * (kx * kx + ky * ky)
        nu4 = 1.0 / (wv2 ** 2 * nsteps * dt)
        beta = 0.5 * wv2 / (2 * np.pi / L * kx) / (nsteps * dt)
        o = orc.QGOracle(nx=N, L=L, dt=dt, use_filter=False, nu4=nu4, nu=0., mu=0., beta=beta, U=0.03)
        o.set_q(A * np.sin(2 * np.pi / L * (kx * x[None, :] + ky * x[:, None])))
        want0 = plane_wave_coefficient(kx, ky, N, L, A)
        assert abs(o.qh[ky, kx] - want0) <= 1e-13 * abs(want0)
        for _ in range(nsteps):
            o.step()
        f = plane_wave_factor(kx, ky, N, L, nsteps * dt, nu4=nu4, beta=beta, U=0.03)
        assert abs(np.angle(f)) > 0.1 and abs(f) < 0.5                  # the wave has moved and decayed
        assert abs(o.qh[ky, kx] - want0 * f) <= 1e-12 * abs(want0 * f)
        rest = o.qh.copy()
        rest[ky, kx] = 0
        assert np.abs(rest).max() <= 1e-9 * abs(want0 * f)     # the aliased 2K harmonic of the Jacobian, O(A)
