"""Parameter sweeps in one batch: ensemble members with their own physical coefficients.

A member's coefficients reach the step through its own ETDRK4 tables (when they differ between members) and through
the per-member coefficient rows of the inversion, the physical-space products, the stage budgets and the host-side
finalisation of status and diagnostics.  Every member here has an independent reference: a golden vector, the numpy
oracle built with its own keywords, a batch-1 run with its own keywords, or the exact linear evolution of a plane
wave under its own operator."""
import inspect
import logging

import numpy as np
import pytest

from cases import (CASES, case_ics, case_params, diag_check, lamb_params, load_golden, plane_wave_coefficient,
                   plane_wave_factor, rel_l2)
from sweep_cases import member_kw, phi_plane_wave, phi_plane_wave_factor, sweep

pytestmark = pytest.mark.gpu
logging.disable(logging.CRITICAL)

TOL_FIELD = 1e-10
TOL_SCALAR = 1e-9
FAMILY_KEYS = ("U", "f", "N", "m", "nu", "nu4", "mu", "nuw", "nu4w", "muw")
QG_KEYS = ("U", "beta", "nu", "nu4", "mu", "nu4c", "nuc", "muc")


def _cls(model):
    from niwqg_b200 import CoupledModel, UnCoupledModel, YBJModel, QLModel, QGModel
    return {"coupled": CoupledModel, "uncoupled": UnCoupledModel, "ybj": YBJModel, "ql": QLModel,
            "qg": QGModel, "qgc": QGModel}[model].Model


def _oracle(model, kw):
    from oracle import niwqg_oracle as orc
    if model in ("qg", "qgc"):
        return orc.QGOracle(**kw)
    return orc.NIWQGOracle(model=model, **kw)


def _seed(m, ics):
    m.set_q(ics["q"])
    if "c" in ics:
        m.set_c(ics["c"])
    if "phi" in ics:
        m.set_phi(ics["phi"])


def _scalar_names(m):
    if hasattr(m, "passive_scalar"):
        return ("Ke", "cvar") if m.passive_scalar else ("Ke",)
    return ("Ke", "Pw", "Kw")


def _state(m):
    B = m.batch
    s = {"scalars": {k: np.atleast_1d(np.asarray(getattr(m, k), float)) for k in _scalar_names(m)},
         "status": m._h.status(),
         "diag": {k: np.asarray(v["value"], float) for k, v in m.diagnostics.items() if "value" in v},
         "fields": {"q": m.q.reshape(B, m.nx, m.nx)}}
    if not hasattr(m, "passive_scalar"):
        s["fields"]["phi"] = m.phi.reshape(B, m.nx, m.nx)
    elif m.passive_scalar:
        s["fields"]["c"] = m.c.reshape(B, m.nx, m.nx)
    return s


def _column(series, b):
    return series if series.ndim == 1 else series[:, b]


def _assert_member_equals(s, b, one, o=0, what=""):
    """Member b of run s is bit for bit member o of run ``one``."""
    for k in s["fields"]:
        assert np.array_equal(s["fields"][k][b], one["fields"][k][o]), (what, k, b)
    for k in s["scalars"]:
        assert s["scalars"][k][b] == one["scalars"][k][o], (what, k, b)
    assert np.array_equal(s["status"][b], one["status"][o]), (what, b)
    for k in s["diag"]:
        if s["diag"][k].ndim > 1:
            assert np.array_equal(_column(s["diag"][k], b), _column(one["diag"][k], o), equal_nan=True), (what, k, b)


def _check_against_oracle(s, b, o, g=None):
    """Member b of run s against the oracle ``o`` (run): fields, budgets, status and diagnostics."""
    F, sc = s["fields"], s["scalars"]
    assert rel_l2(F["q"][b], o.q) < TOL_FIELD, b
    assert abs(sc["Ke"][b] - o.Ke) <= TOL_SCALAR * abs(o.Ke), b
    if "phi" in F:
        assert rel_l2(F["phi"][b], o.phi) < TOL_FIELD, b
        assert abs(sc["Pw"][b] - o.Pw) <= TOL_SCALAR * max(abs(o.Pw), 1e-3 * abs(o.Kw)), b
        assert abs(sc["Kw"][b] - o.Kw) <= TOL_SCALAR * abs(o.Kw), b
        ost = (o.ke_qg(), o.ke_niw(), o.pe_niw())
    else:
        ost = (o.ke_qg(), 0., 0.)
    if "c" in F:
        assert rel_l2(F["c"][b], o.c) < TOL_FIELD, b
        assert abs(sc["cvar"][b] - o.cvar) <= TOL_SCALAR * abs(o.cvar), b
    st = s["status"]
    for j in range(3):
        assert abs(st[b, j] - ost[j]) <= TOL_SCALAR * max(abs(ost[j]), 1e-3 * abs(ost[1])), (b, j)
    od = {"diag_" + k: v for k, v in o.diagnostics().items()}
    for k, ref in od.items():
        diag_check(k[5:], _column(s["diag"][k[5:]], b), ref, od)


def _run_oracle(model, kw, ics):
    o = _oracle(model, kw)
    o.set_q(ics["q"])
    if "c" in ics:
        o.set_c(ics["c"])
    if "phi" in ics:
        o.set_phi(ics["phi"])
    o.run()
    return o


# ---------------------------------------------------------------------------------------------------------------
# 1. Golden pairs that differ only in their parameters, as the two members of one batch
# ---------------------------------------------------------------------------------------------------------------
PAIRS = [("ql_lamb64_filt", "ql_lamb64_diss"), ("qg_lamb64_filt", "qg_lamb64_beta"),
         ("coupled_lamb64_filt", "coupled_lamb64_diss"), ("uncoupled_lamb64_filt", "uncoupled_lamb64_diss")]


@pytest.mark.parametrize("a,b", PAIRS, ids=["ql", "qg", "coupled", "uncoupled"])
def test_golden_pair_in_one_batch(a, b):
    """Each member matches its own golden case.  The batch runs at member 0's diagnostics cadence; a member whose case
    has another cadence is compared with the oracle run at the batch's cadence instead (UnCoupled's diagnostics ticks
    refresh phix, phiy, so the cadence changes its state, F6).  coupled_lamb64_diss has nu4w != 0 beside a member
    with nu4w = 0."""
    model, kw_a, U0, k0 = case_params(a)
    model_b, kw_b, _, _ = case_params(b)
    assert model == model_b
    keys = QG_KEYS if model in ("qg", "qgc") else FAMILY_KEYS
    assert {k for k in kw_b if kw_b[k] != kw_a.get(k)} - set(keys) <= {"tdiags"}
    from niwqg_b200 import Kernel, QGModel
    C = _cls(model)
    init = QGModel.Model.__init__ if model in ("qg", "qgc") else Kernel.Kernel.__init__
    defaults = {k: p.default for k, p in inspect.signature(init).parameters.items()}
    kw = sweep(kw_a, kw_b, keys, defaults)
    assert any(isinstance(v, list) for v in kw.values())
    m = C(batch=2, **kw)
    ics = case_ics(a, m, U0, k0)
    _seed(m, ics)
    m.run()
    s = _state(m)
    for mb, name in enumerate((a, b)):
        g = load_golden(name)
        assert m.tc == int(g["nsteps"])
        if CASES[name][3] != kw["tdiags"]:
            o = _run_oracle(model, dict(member_kw(kw, mb), tdiags=kw["tdiags"]), ics)
            _check_against_oracle(s, mb, o)
            continue
        F, sc = s["fields"], s["scalars"]
        assert rel_l2(F["q"][mb], g["q"]) < TOL_FIELD, name
        assert abs(sc["Ke"][mb] - g["Ke"]) <= TOL_SCALAR * abs(g["Ke"]), name
        if "phi" in F:
            assert rel_l2(F["phi"][mb], g["phi"]) < TOL_FIELD, name
            assert abs(sc["Pw"][mb] - g["Pw"]) <= TOL_SCALAR * max(abs(g["Pw"]), 1e-3 * abs(g["Kw"])), name
            assert abs(sc["Kw"][mb] - g["Kw"]) <= TOL_SCALAR * abs(g["Kw"]), name
        for k, ref in g.items():
            if k.startswith("diag_"):
                diag_check(k[5:], _column(s["diag"][k[5:]], mb), ref, g)


# ---------------------------------------------------------------------------------------------------------------
# 2. Every sweepable keyword varied: each member against the oracle built with its own keywords
# ---------------------------------------------------------------------------------------------------------------
def _sweep_kw(model, N, nsteps=4, tdiags=2):
    """Keywords of a batch of 4 with every per-member keyword different in every member (m, N and f so that hslash
    differs too; nu4w zero in two members and non-zero in two)."""
    qg = model in ("qg", "qgc")
    kw, U0, k0 = lamb_params(N, True, tdiags, nsteps, qg=qg)
    r = np.array([1.0, 0.6, 1.3, 0.85])
    kw["U"] = list(-U0 * np.array([1.0, 0.5, -0.7, 0.2]))
    kw["nu4"] = list(kw["nu4"] * r)
    kw["nu"] = list(np.array([0.0, 1.0, 5.0, 0.5]) if qg else 20 * r)
    kw["mu"] = [0.0, 1e-8, 2e-8, 5e-9]
    if qg:
        kw["beta"] = [0.0, 2e-11, 1e-11, -1e-11]
        if model == "qgc":
            kw.update(passive_scalar=True, nu4c=list(3.e9 * (128 / N) ** 4 * r[::-1]), nuc=[0.0, 2.0, 0.5, 1.0],
                      muc=[1e-8, 0.0, 3e-8, 2e-8])
    else:
        kw["f"] = list(1e-4 * np.array([1.0, 1.2, 0.8, 1.1]))
        kw["N"] = list(0.01 * np.array([1.0, 0.9, 1.3, 1.05]))
        kw["m"] = list(kw["m"] * np.array([1.0, 1.5, 0.7, 1.2]))
        kw["nuw"] = list(50 * r[::-1])
        kw["nu4w"] = [0.0, 2e11 * (64 / N) ** 4, 1e11 * (64 / N) ** 4, 0.0]
        kw["muw"] = [0.0, 3e-8, 1e-8, 2e-8]
    return kw, U0, k0


def _lamb_ics(model, m, U0, k0, B):
    """Member b: the Lamb dipole scaled by (1 + b/4), shifted by b*N/8 cells; a uniform wave or a tracer wave."""
    from oracle import niwqg_oracle as orc
    N = m.nx
    q = orc.lamb_dipole(m, U=U0, R=2 * np.pi / k0)
    out = {"q": np.stack([(1 + 0.25 * b) * np.roll(q, (b * N // 8, 0), (0, 1)) for b in range(B)])}
    if model == "qgc":
        out["c"] = np.stack([np.exp(1j * (k0 / 5 * m.x + (b + 1) * k0 / 5 * m.y)).real for b in range(B)])
    elif model != "qg":
        out["phi"] = np.stack([(1 + 0.1 * b) * (np.ones_like(q) + 1j) * (2 * U0) / np.sqrt(2) for b in range(B)])
    return out


@pytest.mark.parametrize("model,N", [("coupled", 64), ("uncoupled", 64), ("ybj", 64), ("ql", 64), ("qgc", 64),
                                     ("qg", 128), ("coupled", 128)])
def test_every_member_matches_its_oracle(model, N):
    B = 4
    kw, U0, k0 = _sweep_kw(model, N)
    m = _cls(model)(batch=B, **kw)
    ics = _lamb_ics(model, m, U0, k0, B)
    _seed(m, ics)
    m.run()
    s = _state(m)
    for b in range(B):
        o = _run_oracle(model, member_kw(kw, b), {k: v[b] for k, v in ics.items()})
        assert o.tc == m.tc
        _check_against_oracle(s, b, o)
        # the energy equations close on their own member's diagnosed energies (time-stepping error only)
        d = {k: _column(v, b) for k, v in s["diag"].items()}
        # (bounds 3x the oracle's own closure error with these keywords; the filter removes energy the budgets do
        # not see, and YBJ's Pw budget is approximate)
        assert abs(d["Ke"][-1] - d["ke_qg"][-1]) <= 3e-3 * abs(d["ke_qg"][-1]), b
        if "pe_niw" in d:
            tol = 5e-2 if model == "ybj" else 1e-5
            assert abs(d["Pw"][-1] - d["pe_niw"][-1]) <= tol * max(abs(d["pe_niw"][-1]), 1e-3 * abs(d["ke_niw"][-1])), b


# ---------------------------------------------------------------------------------------------------------------
# 3. Bit for bit against single runs, every model and grid size
# ---------------------------------------------------------------------------------------------------------------
def _need_bytes(model, N, B, swept_eqs):
    per = 23 if model not in ("qg", "qgc") else 13
    tables = 13 if model not in ("qg", "qgc") else 9
    return (per * B + tables + 6 * swept_eqs * B) * 16 * N * N


def _require_memory(model, N, B, swept_eqs=2):
    import torch
    free, _ = torch.cuda.mem_get_info()
    need = _need_bytes(model, N, B, swept_eqs)
    if free < need:
        pytest.skip("%s %d^2 batch %d needs about %.1f GB of device memory, %.1f GB free" % (model, N, B, need / 1e9,
                                                                                         free / 1e9))


def _noise_ics(model, N, B, seed):
    rng = np.random.default_rng(seed)
    q = 1e-5 * (rng.random((B, N, N)) - 0.5)
    if model == "qg":
        return {"q": q}
    phi = np.empty((B, N, N), complex)
    phi.real = 0.14 + 0.01 * (rng.random((B, N, N)) - 0.5)
    phi.imag = 0.14 + 0.01 * (rng.random((B, N, N)) - 0.5)
    return {"q": q, "phi": phi}


def _large_sweep_kw(model, N, B, nsteps=3):
    kw, U0, k0 = lamb_params(N, True, 1, nsteps, qg=model == "qg")
    kw["twrite"] = 10 ** 9
    s = np.linspace(1.0, 0.5, B)
    kw["U"] = list(-U0 * s)
    kw["nu4"] = list(kw["nu4"] * s[::-1])
    if model == "qg":
        kw["beta"] = list(1e-11 * s)
    else:
        kw["m"] = list(kw["m"] * (0.5 + s))
        kw["nuw"] = list(50 * s)
        kw["nu4w"] = [0.0] + [1e11 * (64 / N) ** 4] * (B - 1)     # mixed nu4w = 0 and != 0
        kw["muw"] = list(1e-8 * s)
    return kw


def _run(model, kw, ics, batch, nsteps=3):
    m = _cls(model)(batch=batch, **kw)
    _seed(m, ics)
    for _ in range(nsteps):
        m._step_forward()
    return m


BITWISE = [(mdl, N) for N in (512, 1024, 2048, 4096) for mdl in ("coupled", "uncoupled", "ybj", "ql", "qg")]


@pytest.mark.parametrize("model,N", BITWISE)
def test_members_equal_single_runs_with_their_parameters(model, N):
    """Below 8192^2 a single member takes the same kernels as a batch, so every member of a sweep is bit for bit the
    batch-1 run with its own keywords: fields, budgets, status values and diagnostics.  512^2 steps through CUDA graphs
    and 1024^2 loads its column tiles by TMA.  Member 0 has nu4w = 0 beside members with nu4w != 0: the batch then
    carries lap2phi for every member, and member 0 multiplies it by an exact zero, which changes no bit."""
    B = 2 if N >= 2048 else 3
    _require_memory(model, N, B)
    kw = _large_sweep_kw(model, N, B)
    ics = _noise_ics(model, N, B, seed=N + B)
    m = _run(model, kw, ics, B)
    s = _state(m)
    m._h.close()
    for b in range(B):
        one = _run(model, member_kw(kw, b), {k: v[b] for k, v in ics.items()}, 1)
        _assert_member_equals(s, b, _state(one), what="member %d" % b)
        one._h.close()


@pytest.mark.parametrize("model", ["coupled", "qg", "ybj", "ql"])
def test_8192_sweep_matches_single_runs(model):
    """At 8192^2 a batch of 2 takes the ensemble path (cluster column pass, unfused stage kernels with per-member
    tables); one member takes the split transforms and fused kernels (or col3 for QG): agreement to rounding."""
    N, B = 8192, 2
    _require_memory(model, N, B)
    kw = _large_sweep_kw(model, N, B)
    ics = _noise_ics(model, N, B, seed=8192)
    m = _run(model, kw, ics, B)
    F = {k: m._h.field({"q": "Q", "phi": "PHI"}[k]) for k in (("q",) if model == "qg" else ("q", "phi"))}
    sc = {k: np.atleast_1d(np.asarray(getattr(m, k), float)) for k in _scalar_names(m)}
    m._h.close()
    for b in range(B):
        one = _run(model, member_kw(kw, b), {k: v[b] for k, v in ics.items()}, 1)
        for k in F:
            e = rel_l2(one._h.field({"q": "Q", "phi": "PHI"}[k], 0), F[k][b])
            assert e < 1e-12, (k, b, e)
        for k in ("Ke", "Kw"):
            if k in sc:
                v = float(np.atleast_1d(getattr(one, k))[0])
                assert abs(v - sc[k][b]) <= 1e-12 * abs(sc[k][b]), (k, b)
        one._h.close()


# ---------------------------------------------------------------------------------------------------------------
# 4. Shared and per-member paths agree; members are independent
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", ["coupled", "ybj", "ql", "uncoupled", "qgc"])
def test_equal_lists_equal_scalars(model):
    """Keywords given as lists of equal values run the same as the scalars, bit for bit."""
    B = 3
    kw, U0, k0 = _sweep_kw(model, 64)
    scal = {k: (v[1] if isinstance(v, list) else v) for k, v in kw.items()}
    lists = {k: ([v[1]] * B if isinstance(v, list) else v) for k, v in kw.items()}
    runs = []
    for k in (scal, lists):
        m = _cls(model)(batch=B, **k)
        _seed(m, _lamb_ics(model, m, U0, k0, B))
        m.run()
        runs.append(_state(m))
        m._h.close()
    for b in range(B):
        _assert_member_equals(runs[1], b, runs[0], b, "lists")


@pytest.mark.parametrize("model", ["coupled", "ql", "qgc"])
def test_changing_one_member_leaves_the_others_unchanged(model):
    B = 3
    kw, U0, k0 = _sweep_kw(model, 64)
    kw = {k: (v[:B] if isinstance(v, list) else v) for k, v in kw.items()}
    other = {k: (v[:1] + [v[1] * 1.7 + (1e-9 if k in ("mu", "muw", "muc", "beta") else 0.0)] + v[2:]
                 if isinstance(v, list) else v) for k, v in kw.items()}
    runs = []
    for k in (kw, other):
        m = _cls(model)(batch=B, **k)
        _seed(m, _lamb_ics(model, m, U0, k0, B))
        m.run()
        runs.append(_state(m))
        m._h.close()
    assert not np.array_equal(runs[0]["fields"]["q"][1], runs[1]["fields"]["q"][1])
    for b in (0, 2):
        _assert_member_equals(runs[1], b, runs[0], b, "independence")


# ---------------------------------------------------------------------------------------------------------------
# 5. Exact linear evolution of a plane wave under each member's own operator
# ---------------------------------------------------------------------------------------------------------------
def _modes(N):
    return [(37, N // 2 - 3), (3 * N // 8 + 1, 3 * N // 8 + 1)]


@pytest.mark.parametrize("model,N", [(mdl, N) for N in (2048, 4096, 8192) for mdl in ("qg", "ybj", "coupled")])
def test_plane_wave_per_member_operator(model, N):
    """QG: q = A sin(k x + l y) decays and propagates as a Doppler-shifted Rossby wave with the member's nu4, U, beta.
    YBJ and Coupled with q = 0: phi = A exp(i(k x + l y)) has uniform |phi|^2 and J(phi*, phi) = 0, so phih evolves
    by exp(c t), c = -ikU - nu4w|K|^4 - 0.5 i f |K|^2 / kappa^2 - nuw |K|^2 - muw, with the member's m, N, f, U, nu4w,
    nuw, muw (checked against the oracle in tests/test_sweep_cpu.py)."""
    B = 2
    _require_memory(model, N, B)
    L, dt, nsteps, A = 5e5, 2000., 3, 1e-14 if model == "qg" else 1e-6
    T = nsteps * dt
    modes = _modes(N)
    kk = lambda kx: 2 * np.pi / L * kx
    wv = lambda kx, ky: kk(1) ** 2 * (kx * kx + ky * ky)
    base = dict(nx=N, L=L, dt=dt, tmax=T - 1., use_filter=False, twrite=10 ** 9, tdiags=10 ** 9, batch=B)
    if model == "qg":
        nu4 = [2.0 / (wv(*md) ** 2 * T) * s for md, s in zip(modes, (1.0, 0.5))]
        U = [0.4 / (kk(md[0]) * T) * s for md, s in zip(modes, (1.0, -0.7))]
        beta = [0.5 / (T * kk(kx) / wv(kx, ky)) * s for (kx, ky), s in zip(modes, (1.0, -0.6))]
        m = _cls("qg")(nu=0., mu=0., nu4=nu4, U=U, beta=beta, **base)
        x = (np.arange(N) + 0.5) / N * L
        m.set_q(np.stack([A * np.sin(kk(kx) * x[None, :] + kk(ky) * x[:, None]) for kx, ky in modes]))
        m.step(nsteps)
        for b, (kx, ky) in enumerate(modes):
            qh = m._h.field("QH", b)
            want = plane_wave_coefficient(kx, ky, N, L, A) * plane_wave_factor(kx, ky, N, L, T, nu4=nu4[b],
                                                                               beta=beta[b], U=U[b])
            assert abs(qh[ky, kx] - want) <= 1e-10 * abs(want), (b, qh[ky, kx], want)
            qh[ky, kx] = 0
            assert np.abs(qh).max() <= 1e-9 * abs(want), b
    else:
        f = [1.0e-4, 1.3e-4]
        Nb = [0.01, 0.007]
        # the dispersion turns the wave by 1.5 and 0.8 radians: m from hslash = N^2 / (m^2 f)
        m_ = [float(np.sqrt(Nb[b] ** 2 / (f[b] * ph / (0.5 * wv(*modes[b]) * T)))) for b, ph in enumerate((1.5, 0.8))]
        U = [0.4 / (kk(md[0]) * T) * s for md, s in zip(modes, (1.0, -0.7))]
        nu4w = [0.0, 0.5 / (wv(*modes[1]) ** 2 * T)]
        nuw = [0.3 / (wv(*md) * T) * s for md, s in zip(modes, (1.0, 0.4))]
        muw = [0.2 / T, 0.05 / T]
        m = _cls(model)(nu4=0., nu=0., mu=0., f=f, N=Nb, m=m_, U=U, nu4w=nu4w, nuw=nuw, muw=muw, **base)
        phis, c0 = [], []
        for kx, ky in modes:
            p, c = phi_plane_wave(kx, ky, N, L, A)
            phis.append(p)
            c0.append(c)
        m.set_q(np.zeros((N, N)))
        m.set_phi(np.stack(phis))
        del phis
        m.step(nsteps)
        for b, (kx, ky) in enumerate(modes):
            ph = m._h.field("PHIH", b)
            want = c0[b] * phi_plane_wave_factor(kx, ky, N, L, T, f=f[b], Nb=Nb[b], m=m_[b], U=U[b], nu4w=nu4w[b],
                                                 nuw=nuw[b], muw=muw[b])
            assert abs(ph[ky, kx] - want) <= 1e-10 * abs(want), (b, ph[ky, kx], want)
            ph[ky, kx] = 0
            assert np.abs(ph).max() <= 1e-9 * abs(want), b
    m._h.close()


# ---------------------------------------------------------------------------------------------------------------
# 6. API edges
# ---------------------------------------------------------------------------------------------------------------
def test_keyword_errors_name_the_keyword():
    kw, U0, k0 = lamb_params(64, True, 1, 2)
    C = _cls("coupled")
    with pytest.raises(ValueError, match="nu4w"):
        C(batch=3, **dict(kw, nu4w=[0., 1e11]))
    for k, v in (("dt", [kw["dt"]] * 2), ("L", [kw["L"]] * 2), ("use_filter", [True, False]), ("g", [9.81, 9.8]),
                 ("nx", [64, 64])):
        with pytest.raises(ValueError, match=k):
            C(batch=2, **dict(kw, **{k: v}))
    kq, _, _ = lamb_params(64, True, 1, 2, qg=True)
    Q = _cls("qg")
    with pytest.raises(ValueError, match="beta"):
        Q(batch=2, **dict(kq, beta=[0., 1e-11, 2e-11]))
    with pytest.raises(ValueError, match="passive_scalar"):
        Q(batch=2, **dict(kq, passive_scalar=[True, False]))


def test_per_member_tables_match_the_oracle():
    """Tables of a swept equation have a member axis and match the oracle's tables built with each member's keywords
    (tolerances of tests/test_gpu_parity.py::test_tables_match_reference); a shared equation keeps one table."""
    kw, U0, k0 = _sweep_kw("coupled", 32)
    m = _cls("coupled")(batch=4, **kw)
    assert m.expchw.shape == (4, 32, 32) and m.expch.shape == (4, 32, 32) and m.filtr.shape == (32, 32)
    for b in range(4):
        o = _oracle("coupled", member_kw(kw, b))
        for n in ["expch", "expch_h", "expchw", "expch_hw", "Qh", "Qhw"]:
            ref = getattr(o, n)
            assert np.max(np.abs(getattr(m, n)[b] - ref)) <= 1e-13 * np.max(np.abs(ref)), (n, b)
        for n in ["f0", "fab", "fc", "f0w", "fabw", "fcw"]:
            ref = getattr(o, n)
            assert np.max(np.abs(getattr(m, n)[b] - ref)) <= 1e-7 * np.max(np.abs(ref)), (n, b)
        assert np.max(np.abs(m.filtr - o.filtr)) <= 1e-13 * np.max(np.abs(o.filtr))
    m._h.close()
    kw1 = dict(kw, nuw=50., nu4w=0., muw=0., f=1e-4, N=0.01, m=kw["m"][0], U=-U0)     # phi equation shared
    m = _cls("coupled")(batch=4, **kw1)
    assert m.expchw.shape == (32, 32) and m.expch.shape == (4, 32, 32)
    m._h.close()
    kq, _, _ = _sweep_kw("qgc", 32)
    m = _cls("qgc")(batch=4, **kq)
    assert m._h.field("EXPCHC").shape == (4, 32, 17) and m.expch.shape == (4, 32, 17)
    o = _oracle("qgc", member_kw(kq, 2))
    assert np.max(np.abs(m._h.field("EXPCHC", 2) - o.expchc)) <= 1e-13 * np.max(np.abs(o.expchc))
    m._h.close()


# ---------------------------------------------------------------------------------------------------------------
# 7. Checkpoint
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", ["coupled", "qgc"])
def test_sweep_checkpoint_restores_bit_for_bit(model, tmp_path):
    kw, U0, k0 = _sweep_kw(model, 64, nsteps=6)
    C = _cls(model)
    ref = C(batch=4, **kw)
    _seed(ref, _lamb_ics(model, ref, U0, k0, 4))
    for _ in range(3):
        ref._step_forward()
    path = str(tmp_path / "ck")
    ref.save_checkpoint(path)
    ref.run()
    want = _state(ref)
    back = C.from_checkpoint(path)
    assert isinstance(back.U, np.ndarray) and np.array_equal(back.U, np.asarray(kw["U"]))
    back.run()
    got = _state(back)
    for b in range(4):
        _assert_member_equals(got, b, want, b, "restore")
    for k in want["diag"]:
        assert np.array_equal(got["diag"][k], want["diag"][k], equal_nan=True), k
    wrong = dict(kw, nu4=kw["nu4"][:2] + [kw["nu4"][2] * 2] + kw["nu4"][3:])
    other = C(batch=4, **wrong)
    with pytest.raises(ValueError, match="nu4"):
        other.load_checkpoint(path)
