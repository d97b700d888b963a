"""Lagrangian particles on the GPU (kernels_particles.cuh, niwqg_particles_*, Model.set_particles).

- Oracle parity: the golden-case set-ups at 128^2, every model, waves on and off, against the numpy RK4 driver fed
  with the oracle's own stage fields (tests/particles_ref.py).
- Non-interference: with particles every field, budget and diagnostic is bit for bit the run without them, on the
  natural layout, with CUDA graphs (512^2) and on the split transforms (2048^2, de-interleaved rows).
- Exact physics: inertial circles, uniform mean flow, and the interpolation order in a steady cellular flow.
- Ensembles and sweeps, sampling, checkpoints and argument errors.
"""
import importlib
import logging

import numpy as np
import pytest
from scipy.integrate import solve_ivp

import particles_ref as pr
from cases import CASES, EXTRA, lamb_params, case_ics

logging.disable(logging.CRITICAL)

MODULES = {"coupled": "CoupledModel", "uncoupled": "UnCoupledModel", "ybj": "YBJModel", "ql": "QLModel",
           "qg": "QGModel", "qgc": "QGModel"}
NIW = ("coupled", "uncoupled", "ybj", "ql")


def _cls(kind):
    return importlib.import_module("niwqg_b200." + MODULES[kind]).Model


def _case128(name):
    """(kind, keywords, nsteps, U0, k0) of a golden case, set up at 128^2 (tests/cases.py)."""
    kind, nx, use_filter, tdiags, nsteps, _ = CASES[name]
    qg = kind in ("qg", "qgc")
    kw, U0, k0 = lamb_params(128, use_filter, tdiags, nsteps, qg=qg)
    if kind == "qgc":
        kw.update(passive_scalar=True, nu4c=3.e9, nuc=0)
    kw.update(EXTRA.get(name, {}))
    return kind, kw, nsteps, U0, k0


def _seeds(L, N, P, seed=0):
    """P positions: random over [-L, 2L) (unwrapped), plus cell edges and centres, including negative images."""
    rng = np.random.RandomState(seed)
    xy = rng.rand(P, 2) * 3 * L - L
    dx = L / N
    k = np.arange(16)
    xy[:16] = np.stack([k * 7 * dx, (k * 5 + 0.5) * dx], -1)             # edges in x, centres in y
    xy[16:32] = np.stack([-(k + 0.5) * dx - L, (k * 3) * dx + 2 * L], -1)  # centres / edges of other images
    return xy


def _seed_lamb(m, kind, name, U0, k0, scale=None):
    ics = case_ics(name, m, U0, k0)
    q = ics["q"] if scale is None else np.stack([ics["q"] * s for s in scale])
    m.set_q(q)
    if "phi" in ics:
        m.set_phi(ics["phi"] if scale is None else np.stack([ics["phi"] * (2 - s) for s in scale]))
    if "c" in ics:
        m.set_c(ics["c"])


PARITY = [(n, w) for n in ("coupled_lamb64_filt", "coupled_lamb64_dealias", "uncoupled_lamb64_diss", "ql_lamb64_diss",
                           "ybj_lamb64_filt", "ybj_lamb64_nofilt") for w in (False, True)] + \
         [("qg_lamb64_beta", False), ("qg_scalar64_nofilt", False)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,waves", PARITY)
def test_oracle_parity(name, waves):
    kind, kw, nsteps, U0, k0 = _case128(name)
    m = _cls(kind)(**kw)
    o = pr.NIWRecorder(model=kind, **kw) if kind in NIW else pr.QGRecorder(**kw)
    ics = case_ics(name, o, U0, k0)
    for x in (m, o):
        x.set_q(ics["q"])
        if "phi" in ics:
            x.set_phi(ics["phi"])
        if "c" in ics:
            x.set_c(ics["c"])
    xy0 = _seeds(kw["L"], 128, 1000)
    m.set_particles(xy0, waves=waves)
    got = []
    for _ in range(nsteps):
        m._step_forward()
        got.append(m.particles)
    ref = pr.drive(o, xy0, nsteps, waves=waves)
    err = np.max(np.abs(np.array(got) - ref)) / kw["L"]
    assert err < 1e-10, err
    assert np.median(np.abs(ref[-1] - xy0)[:, 0]) > 0.5 * U0 * kw["dt"]      # the particles did move


def _snapshot(m):
    qg = type(m).__module__.endswith("QGModel")
    names = ("q", "qh", "ph", "u", "v") if qg else ("q", "qh", "ph", "phi", "phih", "phix", "phiy", "u", "v", "q_psi")
    out = {n: getattr(m, n) for n in names}
    out["scalars"] = m._h.scalars()
    out["carry"] = m._h.carry()
    out["diagnostics"] = m._h.scalars("diagnostics")
    out["status"] = m._h.status()
    for k, d in m.diagnostics.items():
        out["diag:" + k] = d.get("value")
    out["t"], out["tc"] = m.t, m.tc
    return out


def _assert_same(a, b):
    assert sorted(a) == sorted(b)
    for k in a:
        x, y = a[k], b[k]
        if x is None or y is None:
            assert x is None and y is None, k
            continue
        assert np.shape(x) == np.shape(y) and np.array_equal(x, y), k


def _run(kind, nx, nsteps, particles=None, waves=False, batch=1, tdiags=1, **over):
    name = {"coupled": "coupled_lamb64_filt", "uncoupled": "uncoupled_lamb64_diss", "ybj": "ybj_lamb64_filt",
            "ql": "ql_lamb64_diss", "qg": "qg_lamb64_beta", "qgc": "qg_scalar64_nofilt"}[kind]
    _, kw, _, U0, k0 = _case128(name)
    q_kw, _, _ = lamb_params(nx, kw["use_filter"], tdiags, nsteps, qg=kind in ("qg", "qgc"))
    kw.update(nx=nx, dt=q_kw["dt"], tdiags=tdiags, twrite=2, tmax=1e30, **over)
    if "nu4" in q_kw:
        kw["nu4"] = q_kw["nu4"]
    m = _cls(kind)(batch=batch, **kw)
    _seed_lamb(m, kind, name, U0, k0, scale=None if batch == 1 else [1 + 0.1 * b for b in range(batch)])
    if particles is not None:
        m.set_particles(particles, waves=waves)
    traj = []
    for _ in range(nsteps):
        m._step_forward()
        if particles is not None:
            traj.append(m.particles)
    return m, np.array(traj)


# 2048^2 runs on the split transforms (NIWQG_SPLIT=1), which only the kernel family has
NONINTERFERENCE = [(k, n) for n in (128, 512) for k in ("coupled", "uncoupled", "ybj", "ql", "qg", "qgc")] + \
                  [(k, 2048) for k in NIW]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,nx", NONINTERFERENCE)
def test_particles_change_nothing(kind, nx, monkeypatch):
    if nx == 2048:
        monkeypatch.setenv("NIWQG_SPLIT", "1")
    nsteps = 3 if nx == 2048 else 5
    xy = _seeds(2 * np.pi * 200e3, nx, 4096, seed=1)
    a, _ = _run(kind, nx, nsteps)
    b, traj = _run(kind, nx, nsteps, particles=xy, waves=kind in NIW)
    _assert_same(_snapshot(a), _snapshot(b))
    assert np.all(np.isfinite(traj)) and np.any(traj[-1] != xy)
    # with the particles removed, a step issues exactly the launches of a step without them
    b.set_particles(None)
    assert b.particles is None
    n0, n1 = a._h.launch_count(), b._h.launch_count()
    a.step(3)
    b.step(3)
    assert a._h.launch_count() - n0 == b._h.launch_count() - n1
    _assert_same(_snapshot(a), _snapshot(b))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["coupled", "ybj", "qg"])
def test_seeding_after_the_graphs_were_captured(kind):
    """512^2 steps run as CUDA graphs from the third step on.  Three runs of 8 steps agree bit for bit: A without graphs
    (per-kernel timing on), B seeded before the first step, C seeded after 4 steps - when its graphs exist - with A's
    positions of that time.  The particle clock follows the model's t."""
    xy = _seeds(2 * np.pi * 200e3, 512, 777, seed=2)
    waves = kind != "qg"
    a, _ = _run(kind, 512, 0)
    a._h.profile(True)
    a.set_particles(xy, waves=waves)
    for _ in range(4):
        a._step_forward()
    mid = a.particles
    for _ in range(4):
        a._step_forward()
    b, _ = _run(kind, 512, 0)
    b.set_particles(xy, waves=waves)
    for _ in range(8):
        b._step_forward()
    c, _ = _run(kind, 512, 4)
    c.set_particles(mid, waves=waves)
    for _ in range(4):
        c._step_forward()
    np.testing.assert_array_equal(a.particles, b.particles)
    np.testing.assert_array_equal(a.particles, c.particles)
    for m in (a, b, c):
        assert m._h.particles()[1] == m.t


@pytest.mark.gpu
def test_coupled_trajectories_do_not_depend_on_tdiags():
    """Agreement to rounding, not bit for bit: a diagnostics tick refreshes phix, phiy (pe_niw, F6) through separate
    transforms, while the step forms them with a shared row pass, so the model's own fields after a tick differ from a
    run without it in the last bit."""
    L = 2 * np.pi * 200e3
    xy = _seeds(L, 128, 500, seed=3)
    _, t1 = _run("coupled", 128, 6, particles=xy, waves=True, tdiags=1)
    _, t3 = _run("coupled", 128, 6, particles=xy, waves=True, tdiags=3)
    assert np.max(np.abs(t1 - t3)) <= 1e-12 * L


def _uniform(kind, nx, f, phi0, dt, batch=1, U=0.0):
    L = 2 * np.pi * 100e3
    m = _cls(kind)(nx=nx, L=L, dt=dt, f=f, U=U, batch=batch, use_filter=False, tmax=1e30, twrite=10 ** 9,
                   tdiags=10 ** 9)
    m.set_q(np.zeros((nx, nx)))
    m.set_phi(np.full((nx, nx), phi0, np.complex128))
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("kind", NIW)
def test_inertial_circles(kind):
    f, dt, phi0, n = 1.e-4, 1000.0, 0.3 - 0.4j, 150
    R = abs(phi0) / f
    rng = np.random.RandomState(4)
    xy = (rng.rand(64, 2) - 0.5) * 4 * R                 # near the origin: positions of size R keep their ulp small
    m = _uniform(kind, 64, f, phi0, dt)
    m.set_particles(xy, waves=True)
    zs = [xy[:, 0] + 1j * xy[:, 1]]
    for _ in range(n):
        m.step(1)
        p = m.particles
        zs.append(p[:, 0] + 1j * p[:, 1])
    zs = np.array(zs)                                      # (n + 1, P)
    simpson = np.array([pr.inertial_simpson(z0, phi0, f, dt, n) for z0 in zs[0]]).T
    assert np.max(np.abs(zs - simpson)) < 1e-12 * R
    exact = np.array([pr.inertial_circle(z0, phi0, f, dt * np.arange(n + 1)) for z0 in zs[0]]).T
    bound = np.arange(n + 1)[:, None] * (f * dt) ** 5 / 1440.0 * R
    assert np.all(np.abs(zs - exact) <= bound + 1e-12 * R)
    c = zs[0] - 1j * phi0 / f                              # centres
    ang = np.unwrap(np.angle(zs - c), axis=0)
    assert np.all(np.diff(ang, axis=0) < 0)                # clockwise
    # without the wave velocity the particles stay put (u = v = 0, U = 0)
    m2 = _uniform(kind, 64, f, phi0, dt)
    m2.set_particles(xy, waves=False)
    m2.step(20)
    assert np.max(np.abs(m2.particles - xy)) < 1e-12 * R


@pytest.mark.gpu
def test_inertial_circles_in_an_f_sweep():
    fs, dt, phi0, n = np.array([1.e-4, 1.7e-4, 0.6e-4]), 800.0, 0.25 + 0.1j, 200
    m = _uniform("coupled", 64, fs, phi0, dt, batch=3)
    xy = np.zeros((3, 8, 2))
    xy[:, :, 0] = np.linspace(-500, 500, 8)
    m.set_particles(xy, waves=True)
    m.step(n)
    got = m.particles
    for b, f in enumerate(fs):
        R = abs(phi0) / f
        for j in range(8):
            z = pr.inertial_simpson(complex(*xy[b, j]), phi0, f, dt, n)[-1]
            assert abs(complex(*got[b, j]) - z) < 1e-12 * R, (b, j)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["coupled", "uncoupled", "ybj", "ql", "qg"])
def test_uniform_mean_flow(kind):
    Us = np.array([0.2, -0.13, 0.05])
    L, nx, dt, n = 1.0e6, 64, 3000.0, 40
    kw = dict(nx=nx, L=L, dt=dt, U=Us, batch=3, use_filter=False, tmax=1e30, twrite=10 ** 9, tdiags=10 ** 9)
    m = _cls(kind)(**kw)
    m.set_q(np.zeros((nx, nx)))
    if kind in NIW:
        m.set_phi(np.zeros((nx, nx), np.complex128))
    xy = _seeds(L, nx, 200, seed=6)
    m.set_particles(xy)
    m.step(n)
    got = m.particles
    for b, U in enumerate(Us):
        np.testing.assert_allclose(got[b, :, 0], xy[:, 0] + U * dt * n, rtol=0, atol=1e-12 * L)
        np.testing.assert_array_equal(got[b, :, 1], xy[:, 1])


def _cellular_error(nx, dt, n, xy, A, L):
    kk = 2 * np.pi / L
    m = _cls("qg")(nx=nx, L=L, dt=dt, U=0.0, beta=0.0, nu4=0.0, nu=0.0, mu=0.0, use_filter=False, tmax=1e30,
                    twrite=10 ** 9, tdiags=10 ** 9)
    psi = A * np.sin(kk * m.x) * np.sin(kk * m.y)
    m.set_q(-2 * kk * kk * psi)
    m.set_particles(xy)
    m.step(n)
    got = m.particles

    def rhs(t, z):
        x, y = z[0::2], z[1::2]
        out = np.empty_like(z)
        out[0::2] = -A * kk * np.sin(kk * x) * np.cos(kk * y)
        out[1::2] = A * kk * np.cos(kk * x) * np.sin(kk * y)
        return out

    sol = solve_ivp(rhs, (0.0, n * dt), xy.ravel(), method="DOP853", rtol=1e-12, atol=1e-7)
    ref = sol.y[:, -1].reshape(-1, 2)
    return float(np.max(np.abs(got - ref)))


@pytest.mark.gpu
def test_steady_cellular_flow_converges_at_fourth_order():
    """QG psi = A sin(kx) sin(ky) is steady without dissipation (q is proportional to psi).  Interpolation errors are
    O(dx^4): the trajectory error against an accurate ODE solution of the analytic field must fall by >= 10x per
    doubling of N, at a dt where halving it changes the error by < 1 %."""
    L, A = 1.0e6, 1.6e4
    rng = np.random.RandomState(7)
    xy = rng.rand(64, 2) * L
    dt, n = 5000.0, 400
    errs = [_cellular_error(N, dt, n, xy, A, L) for N in (64, 128, 256)]
    assert errs[0] / errs[1] >= 10 and errs[1] / errs[2] >= 10, errs
    half = _cellular_error(256, dt / 2, 2 * n, xy, A, L)
    assert abs(half - errs[2]) < 0.01 * errs[2], (half, errs[2])


@pytest.mark.gpu
@pytest.mark.parametrize("nx,batch", [(512, 8), (2048, 2)])
def test_members_equal_their_single_runs(nx, batch):
    L = 2 * np.pi * 200e3
    Us = -0.1 * (1 + 0.2 * np.arange(batch))
    fs = 1.e-4 * (1 + 0.1 * np.arange(batch))
    rng = np.random.RandomState(8)
    xy = rng.rand(batch, 600, 2) * 2 * L - 0.5 * L
    ens, traj = _run("coupled", nx, 3, particles=xy, waves=True, batch=batch, U=Us, f=fs)
    for b in range(batch):
        name = "coupled_lamb64_filt"
        _, kw, _, U0, k0 = _case128(name)
        q_kw, _, _ = lamb_params(nx, True, 1, 3)
        kw.update(nx=nx, dt=q_kw["dt"], nu4=q_kw["nu4"], tdiags=1, twrite=2, tmax=1e30, U=Us[b], f=fs[b])
        m = _cls("coupled")(**kw)
        ics = case_ics(name, m, U0, k0)
        s = 1 + 0.1 * b
        m.set_q(ics["q"] * s)
        m.set_phi(ics["phi"] * (2 - s))
        m.set_particles(xy[b], waves=True)
        for _ in range(3):
            m._step_forward()
        np.testing.assert_array_equal(m.particles, traj[-1][b])


@pytest.mark.gpu
def test_perturbing_one_member_leaves_the_others():
    xy = _seeds(2 * np.pi * 200e3, 128, 300, seed=9)
    xy = np.stack([xy, xy + 1000.0, xy - 3000.0])
    _, t0 = _run("ql", 128, 4, particles=xy, waves=True, batch=3)
    xy2 = xy.copy()
    xy2[0] += 12345.0
    _, t1 = _run("ql", 128, 4, particles=xy2, waves=True, batch=3)
    np.testing.assert_array_equal(t0[:, 1:], t1[:, 1:])
    assert np.all(t0[:, 0] != t1[:, 0])


def _require_memory(N, B):
    import torch
    free, _ = torch.cuda.mem_get_info()
    need = (23 * B + 13) * 16 * N * N
    if free < need:
        pytest.skip("coupled %d^2 batch %d needs about %.1f GB of device memory, %.1f GB free"
                    % (N, B, need / 1e9, free / 1e9))


@pytest.mark.gpu
def test_8192_split_path_agrees_with_the_cluster_path():
    """One member at 8192^2 runs the split transforms and fused spectral kernels on de-interleaved physical rows; a
    batch of 2 runs the cluster kernels on the natural layout.  Their trajectories agree to rounding."""
    N, L = 8192, 2 * np.pi * 200e3
    xy = _seeds(L, N, 20000, seed=10)
    _require_memory(N, 2)
    two, t2 = _run("coupled", N, 2, particles=xy, waves=True, batch=2, tdiags=10 ** 9)
    del two
    one, t1 = _run("coupled", N, 2, particles=xy, waves=True, tdiags=10 ** 9)
    assert one._h.particles_count() == 20000
    err = np.max(np.abs(t1[-1] - t2[-1][0])) / L
    assert err < 1e-12, err


@pytest.mark.gpu
@pytest.mark.parametrize("split", ["0", "1"])
@pytest.mark.parametrize("kind", ["coupled", "ybj"])
def test_sampling_matches_the_attribute_arrays(kind, split, monkeypatch):
    monkeypatch.setenv("NIWQG_SPLIT", split)
    nx = 2048
    xy = _seeds(2 * np.pi * 200e3, nx, 3000, seed=11)
    m, _ = _run(kind, nx, 2, particles=xy, waves=True)
    L = m.L
    p = m.particles
    for name in ("q", "u", "v", "phi"):
        got = m.sample_particles(name)
        ref = pr.interp(getattr(m, name), p, L)
        scale = np.max(np.abs(getattr(m, name)))
        assert np.max(np.abs(got - ref)) <= 1e-13 * scale, name
    qg, _ = _run("qg", 256, 2, particles=xy)
    for name in ("q", "u", "v"):
        ref = pr.interp(getattr(qg, name), qg.particles, L)
        assert np.max(np.abs(qg.sample_particles(name) - ref)) <= 1e-13 * np.max(np.abs(getattr(qg, name)))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["coupled", "ybj", "qgc"])
def test_checkpoint_resume_is_exact_for_particles(kind, tmp_path):
    xy = _seeds(2 * np.pi * 200e3, 128, 400, seed=12)
    waves = kind != "qgc"
    ref, traj = _run(kind, 128, 6, particles=xy, waves=waves)
    b, _ = _run(kind, 128, 3, particles=xy, waves=waves)
    b.save_checkpoint(str(tmp_path / "ck"))
    dirty, _ = _run(kind, 128, 4, particles=xy[:7] + 5.0, waves=False)
    dirty.load_checkpoint(str(tmp_path / "ck"))
    for _ in range(3):
        dirty._step_forward()
    np.testing.assert_array_equal(dirty.particles, traj[-1])
    assert dirty._h.particles()[1] == ref._h.particles()[1]
    c = type(ref).from_checkpoint(str(tmp_path / "ck"))
    for _ in range(3):
        c._step_forward()
    np.testing.assert_array_equal(c.particles, traj[-1])
    _assert_same(_snapshot(c), _snapshot(ref))
    # a checkpoint without particles: no PARTICLES.npy, and loading it removes the particles of the model
    nop, _ = _run(kind, 128, 2)
    nop.save_checkpoint(str(tmp_path / "nop"))
    assert not (tmp_path / "nop" / "PARTICLES.npy").exists()
    dirty.load_checkpoint(str(tmp_path / "nop"))
    assert dirty.particles is None


@pytest.mark.gpu
def test_errors():
    m, _ = _run("coupled", 64, 1)
    with pytest.raises(ValueError):
        m.set_particles(np.zeros((5, 3)))
    with pytest.raises(ValueError):
        m.set_particles(np.array([[0.0, np.inf]]))
    with pytest.raises(ValueError):
        m.sample_particles("q")
    qg, _ = _run("qg", 64, 1)
    with pytest.raises(ValueError):
        qg.set_particles(np.zeros((5, 2)), waves=True)
    with pytest.raises(ValueError):
        qg.sample_particles("phi")
    # the library checks its input as well: waves without a wave field, non-finite positions or clock, a bad count
    h = qg._h
    with pytest.raises(RuntimeError, match="wave field"):
        h.particles_set(np.zeros((1, 4, 2)), 0.0, True)
    bad = np.zeros((1, 4, 2))
    bad[0, 2, 1] = np.nan
    with pytest.raises(RuntimeError, match="finite"):
        h.particles_set(bad, 0.0, False)
    with pytest.raises(RuntimeError, match="finite"):
        h.particles_set(np.zeros((1, 4, 2)), float("inf"), False)
    assert h.lib.niwqg_particles_set(h.h, bad.ctypes.data, -1, 0.0, 0, 0) != 0
    assert h.particles_count() == 0
    with pytest.raises(RuntimeError, match="no particles"):
        h.particles_sample("Q")
