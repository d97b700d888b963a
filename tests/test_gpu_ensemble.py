"""Ensembles (batch > 1) against independent references, for every model and grid size.

Batch > 1 is not the single-member code with a loop around it: it turns the split transforms and the three-pass
column transform off (so 8192^2 runs the full-grid cluster column pass and the unfused stage kernels), every kernel
finds its member from blockIdx.y (with different member strides for QG's physical and half-spectrum arrays), the
1024^2 column pass loads its tiles by TMA from a tensor map spanning all members, and every reduction is per member.
Each member here has its own initial condition and its own reference: a golden vector, the numpy oracle, a
single-member run, or an exact transform (a whole-cell shift) of another member."""
import functools
import logging

import numpy as np
import pytest

from cases import (CASES, case_ics, case_params, diag_check, lamb_params, load_golden, plane_wave_coefficient,
                   plane_wave_factor, rel_l2)

pytestmark = pytest.mark.gpu
logging.disable(logging.CRITICAL)

TOL_FIELD = 1e-10      # as tests/test_gpu_parity.py
TOL_SCALAR = 1e-9
TOL_SHIFT = 1e-12      # a member against another member shifted by whole cells: rounding only


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
    """set_q, then set_c, then set_phi: the order of tests/test_gpu_parity.build_cuda (set_q inverts with the phi
    that exists at that time)."""
    m.set_q(ics["q"])
    if "c" in ics:
        m.set_c(ics["c"])
    if "phi" in ics:
        m.set_phi(ics["phi"])


def _scalar_names(m):
    if hasattr(m, "passive_scalar"):
        return ("Ke", "cvar") if m.passive_scalar else ("Ke",)
    return ("Ke", "Pw", "Kw")


def _state(m, fields=True):
    """Everything a run leaves behind, with a leading member axis: fields, budgets, status values
    (ke, kew, pew, cfl) and the diagnostics series ((ticks,) for time, (ticks, B) for the others)."""
    B = m.batch
    s = {"scalars": {k: np.atleast_1d(np.asarray(getattr(m, k), float)) for k in _scalar_names(m)},
         "status": m._h.status(),
         "diag": {k: np.asarray(v["value"], float) for k, v in m.diagnostics.items() if "value" in v}}
    if fields:
        s["fields"] = {"q": m.q.reshape(B, m.nx, m.nx)}
        if not hasattr(m, "passive_scalar"):
            s["fields"]["phi"] = m.phi.reshape(B, m.nx, m.nx)
        elif m.passive_scalar:
            s["fields"]["c"] = m.c.reshape(B, m.nx, m.nx)
    return s


def _column(series, b):
    return series if series.ndim == 1 else series[:, b]


def _member_diags(s, b):
    return {k: _column(v, b) for k, v in s["diag"].items()}


def _budget_scale(name, sc, b=0):
    if name == "Pw":
        return max(abs(sc["Pw"][b]), 1e-3 * abs(sc["Kw"][b]))
    return abs(sc[name][b])


def _close(m):
    m._h.close()


# ---------------------------------------------------------------------------------------------------------------
# 1. A golden member in the middle of every golden case
# ---------------------------------------------------------------------------------------------------------------
def _other_ics(ics, N, seed=5):
    """A different condition for member 0: the dipole (or random field) of the opposite sign plus seeded noise."""
    rng = np.random.RandomState(seed)
    out = {"q": -ics["q"] + 1e-2 * np.abs(ics["q"]).max() * rng.randn(N, N)}
    if "phi" in ics:
        a = np.abs(ics["phi"]).max()
        out["phi"] = (0.6 - 0.3j) * ics["phi"] + 1e-2 * a * (rng.randn(N, N) + 1j * rng.randn(N, N))
    if "c" in ics:
        out["c"] = 0.5 * ics["c"].T + 1e-2 * rng.randn(N, N)
    return out


GOLDEN_SHIFT = lambda N: (N // 4, N // 8)


def _golden_ensemble(name, scale0=1., **over):
    """The batch-3 ensemble of a golden case: member 0 its own condition (times scale0), member 1 the case's
    condition, member 2 that condition shifted by whole cells."""
    model, kw, U0, k0 = case_params(name, **over)
    N = kw["nx"]
    m = _cls(model)(batch=3, **kw)
    ics = case_ics(name, m, U0, k0)
    ic0 = _other_ics(ics, N)
    ic2 = {k: np.roll(v, GOLDEN_SHIFT(N), (0, 1)) for k, v in ics.items()}
    _seed(m, {k: np.stack([scale0 * ic0[k], ics[k], ic2[k]]) for k in ics})
    return m, model, kw, ic0


@pytest.mark.parametrize("name", sorted(CASES))
def test_golden_member_in_an_ensemble(name):
    g = load_golden(name)
    m, model, kw, ic0 = _golden_ensemble(name)
    qg = model in ("qg", "qgc")
    N = kw["nx"]
    shifts = {1: (0, 0), 2: GOLDEN_SHIFT(N)}
    roll = lambda a, b: np.roll(a, shifts[b], (0, 1))
    m._step_forward()
    Q = m.q
    for b in (1, 2):
        assert rel_l2(Q[b], roll(g["q_1"], b)) < TOL_FIELD, b
    if not qg:
        P = m.phi
        for b in (1, 2):
            assert rel_l2(P[b], roll(g["phi_1"], b)) < TOL_FIELD, b
    while m.t < m.tmax:
        m._step_forward()
    assert m.tc == int(g["nsteps"])
    s = _state(m)
    F, sc = s["fields"], s["scalars"]
    for b in (1, 2):
        assert rel_l2(F["q"][b], roll(g["q"], b)) < TOL_FIELD, b
        assert abs(sc["Ke"][b] - g["Ke"]) <= TOL_SCALAR * abs(g["Ke"]), b
        if not qg:
            assert rel_l2(F["phi"][b], roll(g["phi"], b)) < TOL_FIELD, b
            assert abs(sc["Pw"][b] - g["Pw"]) <= TOL_SCALAR * max(abs(g["Pw"]), 1e-3 * abs(g["Kw"])), b
            assert abs(sc["Kw"][b] - g["Kw"]) <= TOL_SCALAR * abs(g["Kw"]), b
        if "c" in g:
            assert rel_l2(F["c"][b], roll(g["c"], b)) < TOL_FIELD, b
            assert abs(sc["cvar"][b] - g["cvar"]) <= TOL_SCALAR * abs(g["cvar"]), b
        d = _member_diags(s, b)
        for k, ref in g.items():
            if k.startswith("diag_"):
                diag_check(k[5:], d[k[5:]], ref, g)
    # the shifted member has the same status values (ke, kew, pew, cfl) as the unshifted one
    st = s["status"]
    for j in range(4):
        assert abs(st[2, j] - st[1, j]) <= TOL_SHIFT * max(abs(st[1, j]), 1e-3 * abs(st[1, 1])), j
    # member 0 against the oracle stepped from its own condition
    o = _oracle(model, kw)
    o.set_q(ic0["q"])
    if "c" in ic0:
        o.set_c(ic0["c"])
    if "phi" in ic0:
        o.set_phi(ic0["phi"])
    o.run()
    assert o.tc == m.tc
    assert rel_l2(F["q"][0], o.q) < TOL_FIELD
    assert abs(sc["Ke"][0] - o.Ke) <= TOL_SCALAR * abs(o.Ke)
    if not qg:
        assert rel_l2(F["phi"][0], o.phi) < TOL_FIELD
        assert abs(sc["Pw"][0] - o.Pw) <= TOL_SCALAR * max(abs(o.Pw), 1e-3 * abs(o.Kw))
        assert abs(sc["Kw"][0] - o.Kw) <= TOL_SCALAR * abs(o.Kw)
        ost = (o.ke_qg(), o.ke_niw(), o.pe_niw())
    else:
        ost = (o.ke_qg(), 0., 0.)
    if "c" in ic0:
        assert rel_l2(F["c"][0], o.c) < TOL_FIELD
        assert abs(sc["cvar"][0] - o.cvar) <= TOL_SCALAR * abs(o.cvar)
    for j in range(3):      # ke, kew, pew of the final state (the cfl column is covered by the member comparisons)
        assert abs(st[0, j] - ost[j]) <= TOL_SCALAR * max(abs(ost[j]), 1e-3 * abs(ost[1])), j
    od = {"diag_" + k: v for k, v in o.diagnostics().items()}
    d = _member_diags(s, 0)
    for k, ref in od.items():
        diag_check(k[5:], d[k[5:]], ref, od)


# ---------------------------------------------------------------------------------------------------------------
# 2. Members are independent
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["coupled_lamb64_diss", "qg_scalar64_nofilt"])
def test_members_are_independent(name):
    """Member 0 scaled by 10^3 (far outside the CFL limit, so no status check: twrite is out of reach) leaves
    members 1 and 2 bit for bit unchanged: fields, budgets, status values and diagnostics."""
    runs = []
    for scale0 in (1., 1e3):
        m = _golden_ensemble(name, scale0=scale0, twrite=10 ** 9)[0]
        m.run()
        runs.append(_state(m))
    a, b = runs
    assert not np.array_equal(a["fields"]["q"][0], b["fields"]["q"][0])
    for k in a["fields"]:
        assert np.array_equal(a["fields"][k][1:], b["fields"][k][1:]), k
    for k in a["scalars"]:
        assert np.array_equal(a["scalars"][k][1:], b["scalars"][k][1:]), k
    assert np.array_equal(a["status"][1:], b["status"][1:])
    for k in a["diag"]:
        assert np.array_equal(a["diag"][k][..., 1:] if a["diag"][k].ndim > 1 else a["diag"][k],
                              b["diag"][k][..., 1:] if b["diag"][k].ndim > 1 else b["diag"][k]), k


# ---------------------------------------------------------------------------------------------------------------
# 3. The measured ensemble sizes: every member a whole-cell shift of member 0
# ---------------------------------------------------------------------------------------------------------------
def _red_noise(N, L, k0, rng):
    """Real field with the McWilliams (1984) red spectrum around k0 and random phases, normalised to max |q| = 1."""
    k = 2 * np.pi / L * np.fft.fftfreq(N, 1. / N)
    wv2 = k[None, :] ** 2 + k[:, None] ** 2
    amp = np.zeros_like(wv2)
    nz = wv2 != 0
    amp[nz] = wv2[nz] / np.sqrt(wv2[nz] * (1. + (wv2[nz] / k0 ** 2) ** 2))
    q = np.fft.ifft2(amp * np.exp(2j * np.pi * rng.rand(N, N))).real
    return q / np.abs(q).max()


def _shifted_ics(model, N, B, kw, k0, U0):
    """Member 0: a random-spectrum q (and a non-uniform phi or c); member b: member 0 shifted by _shift(b)."""
    rng = np.random.RandomState(17)
    L = kw["L"]
    x = (np.arange(N) + 0.5) / N * L
    X, Y = np.meshgrid(x, x)
    ic = {"q": 0.5 * U0 * k0 * _red_noise(N, L, k0, rng)}
    smooth = 1 + 0.5 * np.cos(3 * 2 * np.pi * X / L) + 0.3 * np.sin(2 * 2 * np.pi * Y / L)
    if model == "qgc":
        ic["c"] = smooth + 0.1 * _red_noise(N, L, k0, rng)
    elif model != "qg":
        ic["phi"] = (1 + 1j) * 0.14 * smooth + 0.01 * (_red_noise(N, L, k0, rng) + 1j * _red_noise(N, L, k0, rng))
    return ic, {k: np.stack([np.roll(v, _shift(b, B, N), (0, 1)) for b in range(B)]) for k, v in ic.items()}


def _shift(b, B, N):
    """(b % s, b // s) * N / s cells with s the power of two at or above sqrt(B): (b % 16, b // 16) * N / 16 for 256."""
    s = 1 << (((B - 1).bit_length() + 1) // 2)
    return ((b % s) * N // s, (b // s) * N // s)


def _shifted_model_kw(model, N, nsteps):
    qg = model in ("qg", "qgc")
    kw, U0, k0 = lamb_params(N, True, 1, nsteps, qg=qg)
    kw["twrite"] = 10 ** 9
    if model == "qgc":
        kw.update(passive_scalar=True, nu4c=3.e9 * (128 / N) ** 4, nuc=0)
    return kw, U0, k0


def _check_shifted_members(s, B, N):
    F, sc, st = s["fields"], s["scalars"], s["status"]
    g0 = {"diag_" + k: v for k, v in _member_diags(s, 0).items()}
    for b in range(1, B):
        sh = _shift(b, B, N)
        for k, v in F.items():
            e = rel_l2(v[b], np.roll(v[0], sh, (0, 1)))
            assert e <= TOL_SHIFT, (k, b, e)
        for k in sc:
            assert abs(sc[k][b] - sc[k][0]) <= TOL_SHIFT * _budget_scale(k, sc), (k, b)
        for j in range(4):
            assert abs(st[b, j] - st[0, j]) <= TOL_SHIFT * max(abs(st[0, j]), 1e-3 * abs(st[0, 1])), (j, b)
        d = _member_diags(s, b)
        for k, ref in g0.items():
            diag_check(k[5:], d[k[5:]], ref, g0, tol=TOL_SHIFT)


def _assert_same_run(s, b, t, tb=0):
    """Member b of state s is bit for bit member tb of state t."""
    for k in s["fields"]:
        assert np.array_equal(s["fields"][k][b], t["fields"][k][tb]), k
    for k in s["scalars"]:
        assert s["scalars"][k][b] == t["scalars"][k][tb], k
    assert np.array_equal(s["status"][b], t["status"][tb])
    for k in s["diag"]:
        assert np.array_equal(_column(s["diag"][k], b), _column(t["diag"][k], tb)), k


def _shifted_ensemble(model, N, B, nsteps=5, oracle_members=()):
    kw, U0, k0 = _shifted_model_kw(model, N, nsteps)
    cls = _cls(model)
    m = cls(batch=B, **kw)
    ic, stacked = _shifted_ics(model, N, B, kw, k0, U0)
    _seed(m, stacked)
    for _ in range(nsteps):
        m._step_forward()
    s = _state(m)
    _close(m)
    _check_shifted_members(s, B, N)
    # member 0 is bit for bit the single-member run
    one = cls(**kw)
    _seed(one, ic)
    for _ in range(nsteps):
        one._step_forward()
    _assert_same_run(s, 0, _state(one))
    _close(one)
    if oracle_members:
        o = _oracle(model, kw)
        o.set_q(ic["q"])
        if "phi" in ic:
            o.set_phi(ic["phi"])
        for _ in range(nsteps):
            o.step_forward()
        for b in oracle_members:
            sh = _shift(b, B, N)
            assert rel_l2(s["fields"]["q"][b], np.roll(o.q, sh, (0, 1))) < 1e-10, b
            assert rel_l2(s["fields"]["phi"][b], np.roll(o.phi, sh, (0, 1))) < 1e-10, b
            for k in ("Ke", "Pw", "Kw"):
                v = getattr(o, k)
                assert abs(s["scalars"][k][b] - v) <= 1e-10 * max(abs(v), 1e-3 * abs(o.Kw)), (k, b)
        od = {"diag_" + k: v for k, v in o.diagnostics().items()}
        d = _member_diags(s, 0)
        for k, ref in od.items():
            diag_check(k[5:], d[k[5:]], ref, od)


def test_coupled_512_ensemble_of_256():
    """BASELINE config 5 size on one GPU: Coupled 512^2, 256 members, 5 steps with tdiags=1, CUDA graphs on.
    Members 0 and 255 against the oracle (member 255 against the oracle's run shifted like the member)."""
    _shifted_ensemble("coupled", 512, 256, oracle_members=(0, 255))


@pytest.mark.parametrize("model", ["uncoupled", "ybj", "ql", "qgc"])
def test_512_ensemble_of_8(model):
    _shifted_ensemble(model, 512, 8)


def test_coupled_1024_ensemble_of_4():
    """1024^2 takes the TMA tile loads in the column pass; the tensor map spans the rows of all members.  (Member 0
    equals the single run bit for bit, and the single run is checked against the oracle at this size in
    tests/test_gpu_large.py.)"""
    _shifted_ensemble("coupled", 1024, 4)


# ---------------------------------------------------------------------------------------------------------------
# 4. Large grids
# ---------------------------------------------------------------------------------------------------------------
def _need_bytes(model, N, B):
    """Device bytes of a handle (niwqg_b200.cu create_impl), rounded up: per member about 23 grid-sized complex
    buffers for the kernel family and 13 for QG; the ETDRK4 tables are shared by the members."""
    per = 23 if model not in ("qg", "qgc") else 13
    tables = 13 if model not in ("qg", "qgc") else 9
    return (per * B + tables) * 16 * N * N


def _require_memory(model, N, B):
    import torch
    free, _ = torch.cuda.mem_get_info()
    need = _need_bytes(model, N, B)
    if free < need:
        pytest.skip("%s %d^2 batch %d needs about %.1f GB of device memory, %.1f GB free" % (model, N, B, need / 1e9,
                                                                                         free / 1e9))


@functools.lru_cache(maxsize=1)
def _noise(N, B, seed):
    """White noise on every mode (Nyquist lines included): q ~ 1e-5, phi = 0.14 (1 + i) + 0.01 noise.  Kept for the
    next model at the same size (generating it is most of the host time at 8192^2)."""
    rng = np.random.default_rng(seed)
    q = 1e-5 * (rng.random((B, N, N)) - 0.5)
    phi = np.empty((B, N, N), complex)
    phi.real = 0.14 + 0.01 * (rng.random((B, N, N)) - 0.5)
    phi.imag = 0.14 + 0.01 * (rng.random((B, N, N)) - 0.5)
    return q, phi


def _noise_ics(model, N, B, seed):
    q, phi = _noise(N, B, seed)
    return {"q": q} if model in ("qg", "qgc") else {"q": q, "phi": phi}


def _large_kw(model, N, nsteps=3):
    kw, U0, k0 = lamb_params(N, True, 1, nsteps, qg=model == "qg")
    kw["twrite"] = 10 ** 9
    return kw


def _run(model, kw, ics, batch, nsteps=3):
    m = _cls(model)(batch=batch, **kw)
    _seed(m, ics)
    for _ in range(nsteps):
        m._step_forward()
    return m


@pytest.mark.parametrize("model,N,B", [("coupled", 2048, 3), ("uncoupled", 2048, 3), ("ybj", 2048, 3),
                                       ("ql", 2048, 3), ("coupled", 4096, 2), ("qg", 4096, 2)])
def test_large_ensemble_members_equal_single_runs(model, N, B):
    """Below 8192^2 a single member takes the same kernels as a batch: every member is bit for bit its own single
    run over 3 steps, fields, budgets, status values and diagnostics."""
    _require_memory(model, N, B)
    kw = _large_kw(model, N)
    ics = _noise_ics(model, N, B, seed=N + B)
    m = _run(model, kw, ics, B)
    s = _state(m)
    _close(m)
    for b in range(B):
        one = _run(model, kw, {k: v[b] for k, v in ics.items()}, 1)
        _assert_same_run(s, b, _state(one))
        _close(one)


@pytest.mark.parametrize("model", ["coupled", "qg", "ybj", "ql"])
def test_8192_ensemble_matches_single_runs_and_repeats(model):
    """At 8192^2 a batch of 2 runs the full-grid cluster column pass and the unfused stage kernels; one member runs
    the split transforms with the fused spectral kernels (kernel family) or the three-pass column transform (QG).
    The two must agree to rounding after 3 steps (tolerances of test_split_transform_path_matches_cluster_path_2048),
    and a second fresh batch-2 run must repeat the first bit for bit (the DSMEM barriers of the cluster pass)."""
    N, B = 8192, 2
    _require_memory(model, N, B)
    kw = _large_kw(model, N)
    ics = _noise_ics(model, N, B, seed=8192)
    m = _run(model, kw, ics, B)
    a = _state(m)
    _close(m)
    m = _run(model, kw, ics, B)
    again = _state(m, fields=False)
    for k in a["fields"]:
        for b in range(B):
            assert np.array_equal(m._h.field({"q": "Q", "phi": "PHI"}[k], b), a["fields"][k][b]), (k, b)
    _close(m)
    for k in a["scalars"]:
        assert np.array_equal(a["scalars"][k], again["scalars"][k]), k
    assert np.array_equal(a["status"], again["status"])
    for k in a["diag"]:
        assert np.array_equal(a["diag"][k], again["diag"][k]), k
    del again
    for b in range(B):
        one = _run(model, kw, {k: v[b] for k, v in ics.items()}, 1)
        for k in a["fields"]:
            e = rel_l2(one._h.field({"q": "Q", "phi": "PHI"}[k], 0), a["fields"][k][b])
            assert e < 1e-12, (k, b, e)
        s1 = _state(one, fields=False)
        _close(one)
        for k in ("Ke", "Kw"):
            if k in a["scalars"]:
                assert abs(s1["scalars"][k][0] - a["scalars"][k][b]) <= 1e-12 * abs(a["scalars"][k][b]), (k, b)
        for k, v in a["diag"].items():
            v = _column(v, b)
            w = _column(s1["diag"][k], 0)
            ok = np.isfinite(v)
            if ok.any():
                assert np.max(np.abs(v[ok] - w[ok])) <= 1e-9 * max(np.max(np.abs(v[ok])), 1e-30), (k, b)


# Plane waves q = A sin(k x + l y), one mode per member: near the y Nyquist line, near the x Nyquist line, on the
# diagonal.  J(psi, q) vanishes for a single plane wave, so ETDRK4 must reproduce qh0 exp(c t) of the linear operator.
def _modes(N):
    return [(37, N // 2 - 3), (N // 2 - 5, 29), (3 * N // 8 + 1, 3 * N // 8 + 1)]


PLANE_CASES = [("coupled", 2048, 3), ("coupled", 4096, 3), ("coupled", 8192, 3),
               ("qg", 2048, 3), ("qg", 4096, 3), ("qg", 8192, 3), ("qg", 8192, 1)]


@pytest.mark.parametrize("model,N,B", PLANE_CASES)
def test_plane_wave_per_member_is_exact(model, N, B):
    """niwqg/tests/test_diffusion.py per member: Coupled with nu4 only (phi = 0) decays each mode by
    exp(-nu4 |K|^4 t); QG with beta != 0 carries each mode as an exactly decaying Rossby wave, amplitude and phase
    from the linear operator (the formula is checked against QGOracle in tests/test_oracle_cpu.py).  QG at 8192^2
    with one member runs the three-pass column transform."""
    _require_memory(model, N, B)
    # small amplitude: the Jacobian vanishes for a plane wave, but its 2K harmonic aliases (near the Nyquist lines) and
    # leaves O(A) relative to the wave in one other mode
    L, dt, nsteps, A = 5e5, 2000., 3, 1e-14
    T = nsteps * dt
    modes = _modes(N)[:B] if B > 1 else _modes(N)[:1]
    wv = lambda kx, ky: (2 * np.pi / L) ** 2 * (kx * kx + ky * ky)
    nu4 = 2.0 / (max(wv(*md) ** 2 for md in modes) * T)           # e^-2 on the fastest-decaying mode
    x = (np.arange(N) + 0.5) / N * L
    qs = np.empty((B, N, N))
    for b, (kx, ky) in enumerate(modes):
        qs[b] = A * np.sin(2 * np.pi / L * kx * x[None, :] + 2 * np.pi / L * ky * x[:, None])
    if model == "qg":
        beta = 0.5 / (T * max(2 * np.pi / L * kx / wv(kx, ky) for kx, ky in modes))   # up to half a radian
        m = _cls("qg")(nx=N, L=L, dt=dt, tmax=T - 1., use_filter=False, nu4=nu4, nu=0., mu=0., beta=beta, U=0.,
                       twrite=10 ** 9, tdiags=10 ** 9, batch=B)
        m.set_q(qs if B > 1 else qs[0])
    else:
        beta = 0.
        m = _cls("coupled")(nx=N, L=L, dt=dt, tmax=T - 1., use_filter=False, nu4=nu4, nu4w=0., nu=0., nuw=0.,
                            twrite=10 ** 9, tdiags=10 ** 9, batch=B)
        m.set_q(qs if B > 1 else qs[0])
        m.set_phi(np.zeros((N, N), complex))
    del qs
    m.step(nsteps)
    for b, (kx, ky) in enumerate(modes):
        qh = m._h.field("QH", b)
        want = plane_wave_coefficient(kx, ky, N, L, A) * plane_wave_factor(kx, ky, N, L, T, nu4=nu4, beta=beta)
        assert abs(qh[ky, kx] - want) <= 1e-10 * abs(want), (b, qh[ky, kx], want)
        qh[ky, kx] = 0
        if model != "qg":
            assert abs(qh[N - ky, N - kx] - np.conj(want)) <= 1e-10 * abs(want), b
            qh[N - ky, N - kx] = 0
        assert np.abs(qh).max() <= 1e-9 * abs(want), b
    _close(m)


# ---------------------------------------------------------------------------------------------------------------
# 5. API edges with batch > 1
# ---------------------------------------------------------------------------------------------------------------
def _small(model, B=3, N=64, nsteps=2):
    kw, U0, k0 = _shifted_model_kw(model, N, nsteps)
    return _cls(model)(batch=B, **kw), kw, U0, k0


@pytest.mark.parametrize("model", ["coupled", "qgc"])
def test_whole_grid_array_seeds_every_member(model):
    m, kw, U0, k0 = _small(model)
    ic = _shifted_ics(model, 64, 1, kw, k0, U0)[0]
    _seed(m, ic)
    one = _cls(model)(**kw)
    _seed(one, ic)
    m.step(2); one.step(2)
    s, t = _state(m), _state(one)
    for b in range(3):
        for k in s["fields"]:
            assert np.array_equal(s["fields"][k][b], t["fields"][k][0]), (k, b)
        for k in s["scalars"]:
            assert s["scalars"][k][b] == t["scalars"][k][0], (k, b)


@pytest.mark.parametrize("model", ["coupled", "qg"])
def test_device_lamb_dipole_in_every_member(model):
    from niwqg_b200 import InitialConditions as ic
    m, kw, U0, k0 = _small(model)
    q = ic.LambDipole(m, U=U0, R=2 * np.pi / k0)
    assert ic.LambDipole(m, U=U0, R=2 * np.pi / k0, on_device=True) is None
    Q, QH = m.q, m.qh
    for b in range(3):
        assert np.max(np.abs(Q[b] - q)) <= 1e-13 * np.max(np.abs(q)), b
        assert np.array_equal(QH[b], QH[0]), b
    one = _cls(model)(**kw)
    one.set_q(q)
    assert np.all(np.abs(m.Ke - one.Ke) <= 1e-13 * abs(one.Ke))


def test_batch_rejects_single_member_operations():
    from niwqg_b200 import InitialConditions as ic
    m = _small("coupled")[0]
    for gen in (ic.McWilliams1984, ic.Danioux2015):
        with pytest.raises(RuntimeError, match="single-member"):
            gen(m, on_device=True)
        with pytest.raises(RuntimeError, match="single-member"):
            gen(m, on_device=True, seed=3)
    for jac in (m.jacobian_psi_q, m.jacobian_psi_phi, m.jacobian_phic_phi):
        with pytest.raises(RuntimeError, match="batch"):
            jac()
    with pytest.raises(RuntimeError, match="batch"):
        _small("qg")[0].jacobian_psi_q()


@pytest.mark.parametrize("model", ["coupled", "qg"])
def test_stage_inputs_with_a_member_axis(model):
    import torch
    m, kw, U0, k0 = _small(model, B=4)
    ref = _small(model, B=4)[0]
    stacked = _shifted_ics(model, 64, 4, kw, k0, U0)[1]
    pinned = {}
    for k, v in stacked.items():
        p = torch.empty(v.shape, dtype=torch.complex128 if np.iscomplexobj(v) else torch.float64).pin_memory().numpy()
        p[...] = v
        pinned[k] = p
    m.stage_inputs(**pinned)
    m.set_q()
    if "phi" in pinned:
        m.set_phi()
    _seed(ref, stacked)
    m.step(2); ref.step(2)
    s, t = _state(m), _state(ref)
    for k in s["fields"]:
        assert np.array_equal(s["fields"][k], t["fields"][k]), k
    for k in s["scalars"]:
        assert np.array_equal(s["scalars"][k], t["scalars"][k]), k


def test_wrong_sizes_raise_value_error():
    m = _small("coupled")[0]
    c = _small("qgc")[0]
    N = 64
    for bad in (np.zeros((2, N, N)), np.zeros((4, N, N)), np.zeros((N, N + 2)), np.zeros(3 * N * N - 1)):
        with pytest.raises(ValueError):
            m.set_q(bad)
        with pytest.raises(ValueError):
            m.set_phi(bad.astype(complex))
        with pytest.raises(ValueError):
            m.stage_inputs(q=bad)
        with pytest.raises(ValueError):
            c.set_c(bad)
