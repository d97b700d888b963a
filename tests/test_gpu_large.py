"""Full-size checks of the CUDA path (BASELINE.json sizes): parity against the oracle at the largest sizes the numpy
oracle finishes in seconds, and size-independent properties at 8192^2 where no CPU reference can run (the
reference cannot even initialise above ~2048^2, SURVEY.md F12)."""
import logging

import numpy as np
import pytest

from cases import lamb_params, rel_l2

pytestmark = pytest.mark.gpu
logging.disable(logging.CRITICAL)


def _pair(model, nx, nsteps, use_filter=True, tdiags=10 ** 9):
    from niwqg_b200 import CoupledModel, YBJModel, QLModel
    from oracle import niwqg_oracle as orc
    kw, U0, k0 = lamb_params(nx, use_filter, tdiags, nsteps)
    kw["twrite"] = 10 ** 9
    cls = {"coupled": CoupledModel, "ybj": YBJModel, "ql": QLModel}[model].Model
    m = cls(**kw)
    o = orc.NIWQGOracle(model=model, **kw)
    np.random.seed(7)
    q = orc.mcwilliams1984(o, k0=k0, E=U0 ** 2 / 2)          # random red spectrum (BASELINE config 3)
    phi = (np.ones_like(q) + 1j) * (2 * U0) / np.sqrt(2)
    for mdl in (m, o):
        mdl.set_q(q); mdl.set_phi(phi)
    return m, o


def _budgets_agree(m, o, tol=1e-10):
    for k in ("Ke", "Pw", "Kw"):
        assert abs(getattr(m, k) - getattr(o, k)) <= tol * max(abs(getattr(o, k)), 1e-3 * abs(o.Kw)), k


@pytest.mark.parametrize("model", ["coupled", "ql"])
def test_1024_random_spectrum_10_steps_matches_oracle(model):
    """BASELINE config 3 family at the largest size the numpy oracle steps in seconds: random red spectrum, 10 steps."""
    m, o = _pair(model, 1024, 10)
    for _ in range(10):
        m._step_forward(); o.step_forward()
    assert rel_l2(m.q, o.q) < 1e-10 and rel_l2(m.phi, o.phi) < 1e-10
    _budgets_agree(m, o)


def test_coupled_512_lamb_100_steps_budget_residuals_match_oracle():
    """BASELINE config 2: CoupledModel Lamb dipole + uniform NIW at 512^2, 100 steps, tdiags=1, energy-budget
    Diagnostics.  Fields to 1e-10, and the budget residuals res_ke / res_pe of examples/LambDipole.py:84-90 (finite
    differences of the diagnosed energies minus the diagnosed conversion terms) match the oracle's."""
    from niwqg_b200 import CoupledModel
    from oracle import niwqg_oracle as orc
    nx, nsteps = 512, 100
    kw, U0, k0 = lamb_params(nx, False, 1, nsteps)
    kw["twrite"] = 10 ** 9
    m = CoupledModel.Model(**kw)
    o = orc.NIWQGOracle(model="coupled", **kw)
    q = orc.lamb_dipole(o, U=U0, R=2 * np.pi / k0)
    phi = (np.ones_like(q) + 1j) * (2 * U0) / np.sqrt(2)
    for mdl in (m, o):
        mdl.set_q(q); mdl.set_phi(phi)
    m.run()
    while o.t < o.tmax:
        o.step_forward()
    assert m.tc == o.tc == nsteps
    assert rel_l2(m.q, o.q) < 1e-10 and rel_l2(m.phi, o.phi) < 1e-10
    _budgets_agree(m, o)
    od = o.diagnostics()

    def residuals(d):
        g = lambda k: np.asarray(d[k]["value"] if isinstance(d[k], dict) else d[k], float)
        t = g("time")
        dt = t[1] - t[0]
        dKE, dPE = np.gradient(g("ke_qg"), dt), np.gradient(g("pe_niw"), dt)
        g1, g2, x1, x2 = g("gamma_r"), g("gamma_a"), g("xi_r"), g("xi_a")
        return dKE - (-g1 - g2 + x1 + x2 + g("ep_psi")), dPE - g1 - g2 - g("chi_phi"), dKE, dPE

    rk, rp, dke, dpe = residuals(m.diagnostics)
    ork, orp, odke, odpe = residuals(od)
    # residuals are small differences of the tendencies: compare on the scale of the tendencies themselves
    assert np.max(np.abs(rk - ork)) <= 1e-9 * np.max(np.abs(odke))
    assert np.max(np.abs(rp - orp)) <= 1e-9 * max(np.max(np.abs(odpe)), 1e-3 * np.max(np.abs(odke)))
    # and the budget closes as in the reference's notebook (examples/LambDipole_CoupledModel.ipynb:426-427)
    assert np.max(np.abs(rk[2:-2])) < 1e-2 * np.max(np.abs(dke))


@pytest.mark.skipif(not __import__("os").environ.get("NIWQG_SLOW_TESTS"), reason="oracle needs ~8 min per model at 2048^2")
@pytest.mark.parametrize("model", ["coupled", "ql"])
def test_2048_random_spectrum_10_steps_matches_oracle(model):
    """BASELINE config 3 at its stated size (set NIWQG_SLOW_TESTS=1; result recorded in profiles/r02_parity_2048.txt)."""
    m, o = _pair(model, 2048, 10)
    for _ in range(10):
        m._step_forward(); o.step_forward()
    eq, ep = rel_l2(m.q, o.q), rel_l2(m.phi, o.phi)
    print("2048^2 %s 10 steps: rel-L2 q %.2e phi %.2e" % (model, eq, ep))
    assert eq < 1e-10 and ep < 1e-10
    _budgets_agree(m, o)


@pytest.mark.parametrize("model", ["coupled", "uncoupled", "ybj", "ql"])
def test_split_transform_path_matches_cluster_path_2048(model, monkeypatch):
    """The split transforms + fused spectral kernels (default at 8192^2; NIWQG_SPLIT=1 forces them at 2048^2) against
    the cluster-kernel path on the same run: all four kernel-family models, 3 steps, fields / budgets / diagnostics."""
    from niwqg_b200 import CoupledModel, UnCoupledModel, YBJModel, QLModel
    cls = {"coupled": CoupledModel, "uncoupled": UnCoupledModel, "ybj": YBJModel, "ql": QLModel}[model].Model
    nx = 2048
    kw, U0, k0 = lamb_params(nx, True, 2, 3)
    kw["twrite"] = 10 ** 9
    rng = np.random.RandomState(3)
    q = 1e-5 * rng.randn(nx, nx)
    phi = (np.ones((nx, nx)) + 1j) * 0.14 + 0.01 * (rng.randn(nx, nx) + 1j * rng.randn(nx, nx))
    res = {}
    for split in ("0", "1"):
        monkeypatch.setenv("NIWQG_SPLIT", split)
        m = cls(**kw)
        m.set_q(q); m.set_phi(phi)
        for _ in range(3):
            m._step_forward()
        res[split] = (m.q, m.phi, m.qh, m.phih, m.Ke, m.Pw, m.Kw, {k: np.array(v["value"]) for k, v in m.diagnostics.items()})
        m._h.close()
    a, b = res["0"], res["1"]
    for i in range(4):
        assert rel_l2(b[i], a[i]) < 1e-12
    for i in (4, 6):
        assert abs(a[i] - b[i]) <= 1e-12 * abs(a[i])
    for k, v in a[7].items():
        v = np.atleast_1d(v).astype(float)
        w = np.atleast_1d(b[7][k]).astype(float)
        ok = np.isfinite(v)
        if v.size and ok.any():
            assert np.max(np.abs(v[ok] - w[ok])) <= 1e-9 * max(np.max(np.abs(v[ok])), 1e-30), k


def test_ybj_2048_random_spectrum_matches_oracle():
    m, o = _pair("ybj", 2048, 3)
    for _ in range(3):
        m._step_forward(); o.step_forward()
    assert rel_l2(m.phi, o.phi) < 1e-10


def test_8192_linear_propagator_is_exact():
    """niwqg/tests/test_diffusion.py at the target grid: with nu4 only and a plane-wave q, phi = 0, ETDRK4 must
    reproduce qh0 * exp(-nu4 wv4 t) (tables, transforms through the cluster kernels, stage kernels at full size)."""
    from niwqg_b200 import CoupledModel
    N = 8192
    kx, ky = 37, 4001            # one mode near the grid scale in y: strong, exactly known decay
    L = 5e5
    k, l = 2 * np.pi * kx / L, 2 * np.pi * ky / L
    nu4 = 2.0 / ((k * k + l * l) ** 2 * 3 * 2000.)          # e^-2 over the three steps
    m = CoupledModel.Model(nx=N, L=L, use_filter=False, nu4=nu4, nu4w=0., nu=0., nuw=0., dt=2000., tmax=3 * 2000. - 1.,
                           twrite=10 ** 9, tdiags=10 ** 9)
    xs = (np.arange(N) + 0.5) / N * m.L
    A = 1e-10                    # small amplitude: the (analytically vanishing) Jacobian's rounding noise stays negligible
    qi = A * np.sin(k * xs[None, :] + l * xs[:, None])
    m.set_q(qi); m.set_phi(np.zeros((N, N), complex))
    m.run()
    assert m.tc == 3
    qh = m.qh
    decay = np.exp(-nu4 * (k * k + l * l) ** 2 * 3 * 2000.)
    # qi = Im exp(i(kx+ly)): modes (ky,kx) and (-ky,-kx) with amplitude N^2/2 and the half-cell phase
    amp = abs(qh[ky, kx]) / (N * N / 2) / A
    assert abs(amp - decay) < 1e-10 * decay, (amp, decay)
    assert abs(abs(qh[N - ky, N - kx]) / (N * N / 2) / A - decay) < 1e-10 * decay
    qh[ky, kx] = 0; qh[N - ky, N - kx] = 0
    assert np.abs(qh).max() < 1e-5 * (N * N / 2) * A * decay
    # and the physical field is the decayed plane wave
    assert rel_l2(m.q, decay * qi) < 1e-6     # the Jacobian rounding noise of all other modes (the reference shows the same)


def test_8192_step_conserves_and_budgets_close():
    """One Coupled step at 8192^2 from the bench initial condition: finite, the integrated budgets follow the diagnosed
    energies, and a second model stepped from the same state agrees bit for bit (deterministic reductions)."""
    from niwqg_b200 import CoupledModel, InitialConditions as ic
    N = 8192
    kw, U0, k0 = lamb_params(N, True, 1, 2)
    kw["twrite"] = 10 ** 9
    m = CoupledModel.Model(**kw)
    q = ic.LambDipole(m, U=U0, R=2 * np.pi / k0)
    phi = (np.ones_like(q) + 1j) * (2 * U0) / np.sqrt(2)
    m.set_q(q); m.set_phi(phi)
    m._step_forward(); m._step_forward()
    d = m.diagnostics
    ke, Ke = d["ke_qg"]["value"], d["Ke"]["value"]
    assert np.all(np.isfinite(ke)) and np.all(np.isfinite(d["ke_niw"]["value"]))
    assert abs(ke[-1] - Ke[-1]) < 1e-6 * ke[0]
    assert abs(d["ke_niw"]["value"][-1] - d["Kw"]["value"][-1]) < 1e-6 * d["ke_niw"]["value"][0]
    q1 = m.q
    del m
    m2 = CoupledModel.Model(**kw)
    m2.set_q(q); m2.set_phi(phi)
    m2._step_forward(); m2._step_forward()
    assert np.array_equal(q1, m2.q)


@pytest.mark.parametrize("N", [2048, 4096, 8192])
def test_cluster_transforms_are_bitwise_repeatable(N):
    """The cluster kernels exchange through distributed shared memory behind barriers; a missing barrier would show up
    as run-to-run differences (compute-sanitizer's racecheck is not available on the GPU pool).  Same input, several
    back-to-back transforms (so different CTA placements and timings), bit-identical outputs, forward and inverse.
    niwqg_fft2 transforms one member, and one member at 8192^2 takes the split transforms (fft2_split), so N = 8192
    here exercises the split path; the full-grid 8192^2 cluster column pass runs only for batch > 1 and is repeated
    bit for bit in tests/test_gpu_ensemble.py::test_8192_ensemble_matches_single_runs_and_repeats."""
    from niwqg_b200 import _native as nat
    h = nat.Handle(model=nat.MODEL_YBJ, nx=N, batch=1, device=0, L=5e5, dt=1e4, f=1e-4, N=0.01, m=0.025, nu=20., nuw=50.)
    rng = np.random.RandomState(11)
    x = rng.randn(N, N) + 1j * rng.randn(N, N)
    X0 = h.fft2(x, nat.FFT_C2C_FWD)
    x0 = h.fft2(X0, nat.FFT_C2C_INV)
    for _ in range(3):
        assert np.array_equal(h.fft2(x, nat.FFT_C2C_FWD), X0)
        assert np.array_equal(h.fft2(X0, nat.FFT_C2C_INV), x0)
    assert rel_l2(x0, x) < 5e-15
    h.close()
