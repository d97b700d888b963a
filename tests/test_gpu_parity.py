"""GPU parity tests (run on the B200 box: ``pytest -m gpu``).  Every call goes through the
C ABI (niwqg_b200/_native.py -> libniwqg_b200.so); the checker is the numpy oracle
(oracle/niwqg_oracle.py) and the golden vectors produced by the unmodified reference
(tests/golden/).  Tolerances: the north-star bar is rel-L2 <= 1e-10 on q and phi after 100
steps (fp64 throughout); budgets are compared relative to their own magnitude."""
import numpy as np
import pytest

from cases import CASES, case_ics, case_params, diag_check, lamb_params, load_golden, rel_l2

pytestmark = pytest.mark.gpu

TOL_FIELD = 1e-10      # BASELINE.json north_star: relative L2 on q and phi
TOL_SCALAR = 1e-9      # integrated budgets Ke, Pw, Kw (relative)


def _models():
    from niwqg_b200 import CoupledModel, UnCoupledModel, YBJModel, QLModel, QGModel
    return {"coupled": CoupledModel.Model, "uncoupled": UnCoupledModel.Model, "ybj": YBJModel.Model,
            "ql": QLModel.Model, "qg": QGModel.Model, "qgc": QGModel.Model}


def build_cuda(name, **over):
    import logging
    logging.disable(logging.CRITICAL)
    model, kw, U0, k0 = case_params(name, **over)
    m = _models()[model](**kw)
    ics = case_ics(name, m, U0, k0)
    m.set_q(ics["q"])
    if "c" in ics:
        m.set_c(ics["c"])
    if "phi" in ics:
        m.set_phi(ics["phi"])
    return m


@pytest.mark.parametrize("N", [32, 64, 128, 256, 512, 1024, 2048])
def test_fft2_matches_numpy(N):
    from niwqg_b200 import _native as nat
    h = nat.Handle(model=nat.MODEL_UNCOUPLED, nx=N, batch=1, device=0, L=5e5, dt=1e4, f=1e-4, N=0.01, m=0.025,
                   nu=20., nuw=50.)
    rng = np.random.RandomState(N)
    x = rng.randn(N, N) + 1j * rng.randn(N, N)
    r = rng.randn(N, N)
    assert rel_l2(h.fft2(x, nat.FFT_C2C_FWD), np.fft.fft2(x)) < 2e-15
    assert rel_l2(h.fft2(x, nat.FFT_C2C_INV), np.fft.ifft2(x)) < 2e-15
    assert rel_l2(h.fft2(r, nat.FFT_R2C), np.fft.rfft2(r)) < 2e-15
    assert rel_l2(h.fft2(r, nat.FFT_R2C_FULL), np.fft.fft2(r)) < 2e-15
    hs = np.fft.rfft2(r)
    hs[3, 0] += 0.5j; hs[5, N // 2] += 0.25j; hs[0, 0] += 1j      # irfft2 must drop these, as numpy does
    assert rel_l2(h.fft2(hs, nat.FFT_C2R), np.fft.irfft2(hs)) < 2e-15
    h.close()


@pytest.mark.parametrize("N", [4096, 8192])
def test_fft2_large_properties(N):
    """Full-size grids: round trip, Parseval and a known-answer plane wave (size-independent properties)."""
    from niwqg_b200 import _native as nat
    h = nat.Handle(model=nat.MODEL_YBJ, nx=N, batch=1, device=0, L=5e5, dt=1e4, f=1e-4, N=0.01, m=0.025,
                   nu=20., nuw=50.)
    rng = np.random.RandomState(1)
    x = rng.randn(N, N) + 1j * rng.randn(N, N)
    X = h.fft2(x, nat.FFT_C2C_FWD)
    assert abs((np.abs(X) ** 2).sum() / N ** 2 - (np.abs(x) ** 2).sum()) / (np.abs(x) ** 2).sum() < 1e-13
    assert rel_l2(h.fft2(X, nat.FFT_C2C_INV), x) < 5e-15
    # rows/columns against numpy's 1-D transforms on a subset
    assert rel_l2(X[:, 5], np.fft.fft(np.fft.fft(x, axis=1)[:, 5])) < 5e-15
    jj, ii = np.meshgrid(np.arange(N), np.arange(N))
    w = np.exp(2j * np.pi * ((7 * jj + 1234 * ii) % N) / N)
    W = h.fft2(w, nat.FFT_C2C_FWD)
    assert abs(W[1234, 7] - N * N) / (N * N) < 1e-13
    W[1234, 7] = 0
    assert np.abs(W).max() / (N * N) < 1e-12
    h.close()


def test_tables_match_reference():
    """ETDRK4 tables + filter generated on the device vs the reference's (niwqg/Kernel.py:400-454, :267-284).
    The contour-mean formulas amplify rounding where |c dt| ~ 1 (both implementations; see DESIGN.md), hence 1e-7."""
    from niwqg_b200 import CoupledModel
    import logging
    logging.disable(logging.CRITICAL)
    g = load_golden("coeffs_coupled32")
    kw, U0, k0 = lamb_params(32, True, 1, 1)
    m = CoupledModel.Model(**kw)
    for n in ["expch", "expch_h", "expchw", "expch_hw", "Qh", "Qhw", "filtr"]:
        assert np.max(np.abs(getattr(m, n) - g[n])) <= 1e-13 * np.max(np.abs(g[n])), n
    # f0, fab, fc: 32-point contour means of (...)/LR^3 with LR = c dt + r_j on the unit circle.  Where the circle
    # passes close to the origin (|c dt| ~ 1) the terms are huge and cancel, and BOTH implementations lose digits
    # there, so the comparison is split: every wavenumber whose contour stays >= 0.1 away from the origin must
    # agree to 1e-13, the others (a thin shell |c dt| ~ 1) to 1e-7; their number and worst error are reported.
    r = np.exp(2j * np.pi * (np.arange(1, 33) / 32.))
    for tabs, cname in ((("f0", "fab", "fc"), "c_q"), (("f0w", "fabw", "fcw"), "c_phi")):
        ch = np.log(g["expch" if cname == "c_q" else "expchw"].astype(complex))     # c dt (principal branch: |Im| < pi here)
        dist = np.min(np.abs(ch[..., None] + r), axis=-1)
        far = dist > 0.1
        assert far.mean() > 0.9
        for n in tabs:
            err = np.abs(getattr(m, n) - g[n]) / np.max(np.abs(g[n]))
            print("%s: %d of %d points within 0.1 of the contour, max err there %.1e, elsewhere %.1e"
                  % (n, (~far).sum(), far.size, err[~far].max() if (~far).any() else 0.0, err[far].max()))
            assert err[far].max() <= 1e-13, n
            assert err.max() <= 1e-7, n


@pytest.mark.parametrize("name", sorted(CASES))
def test_step_parity_against_reference_golden(name):
    g = load_golden(name)
    m = build_cuda(name)
    qg = CASES[name][0] in ("qg", "qgc")
    m._step_forward()
    assert rel_l2(m.q, g["q_1"]) < TOL_FIELD
    if not qg:
        assert rel_l2(m.phi, g["phi_1"]) < TOL_FIELD
    while m.t < m.tmax:
        m._step_forward()
    assert m.tc == int(g["nsteps"])
    eq = rel_l2(m.q, g["q"])
    assert eq < TOL_FIELD, eq
    assert abs(m.Ke - g["Ke"]) <= TOL_SCALAR * abs(g["Ke"])
    if not qg:
        ep = rel_l2(m.phi, g["phi"])
        assert ep < TOL_FIELD, ep
        assert abs(m.Pw - g["Pw"]) <= TOL_SCALAR * max(abs(g["Pw"]), 1e-3 * abs(g["Kw"]))
        assert abs(m.Kw - g["Kw"]) <= TOL_SCALAR * abs(g["Kw"])
    if "c" in g:
        assert rel_l2(m.c, g["c"]) < TOL_FIELD
        assert abs(m.cvar - g["cvar"]) <= TOL_SCALAR * abs(g["cvar"])


@pytest.mark.parametrize("name", ["coupled_lamb64_filt", "coupled_lamb64_nofilt", "uncoupled_lamb64_filt", "ql_lamb64_filt",
                                  "ybj_lamb64_filt", "coupled_rand64_filt", "coupled_lamb128_nofilt_100",
                                  "qg_lamb64_filt", "qg_scalar64_nofilt", "coupled_lamb64_diss", "coupled_lamb64_dealias",
                                  "uncoupled_lamb64_diss", "ql_lamb64_diss", "qg_lamb64_beta"])
def test_diagnostics_series_match_reference(name):
    g = load_golden(name)
    m = build_cuda(name)
    m.run()
    for k, ref in g.items():
        if not k.startswith("diag_"):
            continue
        dn = k[5:]
        diag_check(dn, m.diagnostics[dn]['value'], ref, g)


def test_ensemble_members_match_single_runs():
    """batch > 1 (config 5): members are independent and identical to single runs."""
    import logging
    logging.disable(logging.CRITICAL)
    from niwqg_b200 import CoupledModel
    from oracle import niwqg_oracle as orc
    kw, U0, k0 = lamb_params(64, True, 1000, 5)
    single = CoupledModel.Model(**kw)
    q = orc.lamb_dipole(single, U=U0, R=2 * np.pi / k0)
    rng = np.random.RandomState(3)
    qs = np.stack([q, 0.5 * q + 1e-7 * rng.randn(64, 64), -q])
    phis = np.stack([(np.ones_like(q) + 1j) * a for a in (0.14, 0.07, 0.2)])
    ens = CoupledModel.Model(batch=3, **kw)
    ens.set_q(qs); ens.set_phi(phis)
    ens.step(5)
    Q, P = ens.q, ens.phi
    for b in range(3):
        s = CoupledModel.Model(**kw)
        s.set_q(qs[b]); s.set_phi(phis[b])
        s.step(5)
        assert np.array_equal(s.q, Q[b]) and np.array_equal(s.phi, P[b])


def test_seeding_order_semantics_F5():
    """set_q inverts with the phi that exists at that time; set_phi does not re-invert (Kernel.py:520-551)."""
    import logging
    logging.disable(logging.CRITICAL)
    from niwqg_b200 import CoupledModel
    from oracle import niwqg_oracle as orc
    kw, U0, k0 = lamb_params(64, True, 1000, 1)
    a = CoupledModel.Model(**kw); o = orc.NIWQGOracle(model="coupled", **kw)
    q = orc.lamb_dipole(o, U=U0, R=2 * np.pi / k0)
    phi = (np.ones_like(q) + 1j) * 0.14 * (1 + 0.5 * np.cos(3 * 2 * np.pi * o.x / o.L) + 0.3 * np.sin(2 * 2 * np.pi * o.y / o.L))
    for mdl in (a, o):
        mdl.set_phi(phi); mdl.set_q(q)            # swapped order
    a._step_etdrk4(); o.step()
    assert rel_l2(a.phi, o.phi) < TOL_FIELD and rel_l2(a.q, o.q) < TOL_FIELD
    b = CoupledModel.Model(**kw)
    b.set_q(q); b.set_phi(phi); b._step_etdrk4()
    assert rel_l2(b.phi, o.phi) > 1e-7        # the order matters, as in the reference


@pytest.mark.parametrize("model", ["coupled", "qg"])
def test_run_with_snapshots_generator(model):
    """Kernel.run_with_snapshots (niwqg/Kernel.py:161-181; QGModel.py:175-195): yields t every tsnapint while stepping to
    tmax; the state after the generator is exhausted equals a plain run()."""
    import logging
    logging.disable(logging.CRITICAL)
    from niwqg_b200 import CoupledModel, QGModel
    from oracle import niwqg_oracle as orc
    qg = model == "qg"
    kw, U0, k0 = lamb_params(64, True, 5, 12, qg=qg)
    cls = QGModel.Model if qg else CoupledModel.Model
    a, b = cls(**kw), cls(**kw)
    q = orc.lamb_dipole(a, U=U0, R=2 * np.pi / k0)
    for mdl in (a, b):
        mdl.set_q(q)
        if not qg:
            mdl.set_phi((np.ones_like(q) + 1j) * (2 * U0) / np.sqrt(2))
    snaps = list(a.run_with_snapshots(tsnapstart=0., tsnapint=3 * a.dt))
    b.run()
    assert a.tc == b.tc == 12
    assert np.array_equal(a.q, b.q)
    # reference semantics: yield t after every step with tc % ceil(tsnapint / dt) == 0 (and t >= tsnapstart)
    assert len(snaps) == 4
    assert np.allclose(snaps, np.array([3, 6, 9, 12]) * a.dt, rtol=1e-12)
