"""Checkpoint and exact restart on the GPU (niwqg_b200/Checkpoint.py, niwqg_state_slots / niwqg_set_field / carry).

Run A steps 2n times.  Run B steps n times, saves, and the checkpoint is restored into a different, dirty instance
(seeded from another initial condition and stepped once more than B, so its ping-pong parity is the opposite one and its
carried buffers and ep_psi sums hold other values), which then steps n more times.  Every field attribute, every state
slot, Ke/Pw/Kw, every diagnostics series, t and tc must then be bit-for-bit those of run A."""
import logging
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest

from cases import lamb_params, rel_l2, EXTRA

logging.disable(logging.CRITICAL)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# name: (model module, nx, constructor keywords on top of lamb_params)
CASES = {
    "coupled_filt": ("CoupledModel", 64, dict(use_filter=True)),
    "coupled_nofilt": ("CoupledModel", 64, dict(use_filter=False)),
    "coupled_dealias": ("CoupledModel", 64, dict(use_filter=False, dealias=True)),
    "coupled_diss128": ("CoupledModel", 128, dict(EXTRA["coupled_lamb64_diss"], tdiags=2)),
    "uncoupled_tdiags3": ("UnCoupledModel", 64, dict(tdiags=3)),
    "ybj": ("YBJModel", 64, dict(tdiags=2)),
    "ybj_diss": ("YBJModel", 64, dict(nu4w=2.e11, tdiags=3)),
    "ql_diss": ("QLModel", 64, dict(EXTRA["ql_lamb64_diss"], tdiags=2)),
    "qg": ("QGModel", 64, dict(tdiags=2)),
    "qg_scalar": ("QGModel", 128, dict(tdiags=1, passive_scalar=True, use_filter=False)),
}

FAMILY_FIELDS = ("q", "qh", "ph", "p", "phi", "phih", "phix", "phiy", "lapphi", "u", "v", "q_psi")
QG_FIELDS = ("q", "qh", "ph", "p", "u", "v", "c", "ch")


def _cls(name):
    import importlib
    return importlib.import_module("niwqg_b200." + name).Model


def _kw(case, nsteps=100):
    mod, nx, extra = CASES[case]
    kw, U0, k0 = lamb_params(nx, extra.get("use_filter", True), 1, nsteps, qg=(mod == "QGModel"))
    kw["twrite"] = 3                 # status ticks (phix, phiy refreshed, ke/cfl cached) inside the runs
    kw.update(extra)
    return mod, kw, U0, k0


def _seed(m, mod, U0, k0, variant=0, batch=1):
    """Lamb dipole (variant 0) or another, noisier initial condition (variant 1); one per member when batch > 1."""
    from niwqg_b200 import InitialConditions as ic
    rng = np.random.RandomState(3 + variant)
    q0 = ic.LambDipole(m, U=U0, R=2 * np.pi / k0)
    N = m.nx
    qs = np.stack([q0 * (1 + 0.3 * variant + 0.1 * b) + 0.05 * np.abs(q0).max() * rng.randn(N, N) for b in range(batch)])
    m.set_q(qs[0] if batch == 1 else qs)
    if mod == "QGModel":
        if m.passive_scalar:
            m.set_c(np.cos(2 * np.pi * m.x / m.L) * (1 + 0.1 * rng.randn(N, N)))
        return
    phis = np.stack([(np.ones((N, N)) + 1j) * (2 * U0) / np.sqrt(2) * (1 + 0.1 * rng.randn(N, N)) for _ in range(batch)])
    m.set_phi(phis[0] if batch == 1 else phis)


def _snapshot(m):
    """Everything a user can observe of the model, read once."""
    fields = QG_FIELDS if type(m).__module__.endswith("QGModel") else FAMILY_FIELDS
    if hasattr(m, "qwh"):
        fields = fields + ("qw", "qwh")
    out = {f: getattr(m, f) for f in fields}
    for s in m._h.state_slots():
        out["slot:" + s] = np.stack([m._h.field(s, b) for b in range(m.batch)])
    out["carry"] = m._h.carry()
    for k in ("Ke", "Pw", "Kw", "cvar"):
        if hasattr(type(m), k):
            out[k] = getattr(m, k)
    for k, d in m.diagnostics.items():
        out["diag:" + k] = d.get("value")
    out["t"], out["tc"] = m.t, m.tc
    for k in ("ke", "kew", "pew", "cfl"):
        out["status:" + k] = getattr(m, k, None)
    return out


def _assert_same(a, b):
    assert sorted(a) == sorted(b)
    for k in a:
        x, y = a[k], b[k]
        if x is None or y is None:
            assert x is None and y is None, k
            continue
        assert np.shape(x) == np.shape(y) and np.array_equal(x, y), k


def _run_a(case, n, batch=1):
    mod, kw, U0, k0 = _kw(case)
    a = _cls(mod)(batch=batch, **kw)
    _seed(a, mod, U0, k0, batch=batch)
    for _ in range(2 * n):
        a._step_forward()
    return _snapshot(a)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 4])
@pytest.mark.parametrize("case", sorted(CASES))
def test_exact_resume_into_a_dirty_instance(case, n, tmp_path):
    mod, kw, U0, k0 = _kw(case)
    ref = _run_a(case, n)
    b = _cls(mod)(**kw)
    _seed(b, mod, U0, k0)
    for _ in range(n):
        b._step_forward()
    b.save_checkpoint(str(tmp_path / "ck"))
    dirty = _cls(mod)(**kw)
    _seed(dirty, mod, U0, k0, variant=1)
    for _ in range(n + 1):
        dirty._step_forward()
    dirty.load_checkpoint(str(tmp_path / "ck"))
    for _ in range(n):
        dirty._step_forward()
    _assert_same(_snapshot(dirty), ref)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["coupled_filt", "uncoupled_tdiags3", "ybj", "ql_diss", "qg_scalar"])
def test_save_is_side_effect_free_and_from_checkpoint_resumes(case, tmp_path):
    n = 4
    mod, kw, U0, k0 = _kw(case)
    ref = _run_a(case, n)
    b = _cls(mod)(**kw)
    _seed(b, mod, U0, k0)
    for _ in range(n):
        b._step_forward()
    b.save_checkpoint(str(tmp_path / "ck"))
    b.save_checkpoint(str(tmp_path / "ck"))          # replaces the first one
    for _ in range(n):
        b._step_forward()
    _assert_same(_snapshot(b), ref)
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        c = _cls(mod).from_checkpoint(str(tmp_path / "ck"))
    assert not [w for w in caught if "exactly" in str(w.message)]      # nothing overridden: no exactness warning
    for _ in range(n):
        c._step_forward()
    _assert_same(_snapshot(c), ref)


@pytest.mark.gpu
def test_ensemble_exact_resume(tmp_path):
    n, batch = 3, 3
    mod, kw, U0, k0 = _kw("coupled_filt")
    ref = _run_a("coupled_filt", n, batch=batch)
    b = _cls(mod)(batch=batch, **kw)
    _seed(b, mod, U0, k0, batch=batch)
    for _ in range(n):
        b._step_forward()
    b.save_checkpoint(str(tmp_path / "ck"))
    dirty = _cls(mod)(batch=batch, **kw)
    _seed(dirty, mod, U0, k0, variant=1, batch=batch)
    for _ in range(n + 1):
        dirty._step_forward()
    dirty.load_checkpoint(str(tmp_path / "ck"))
    for _ in range(n):
        dirty._step_forward()
    _assert_same(_snapshot(dirty), ref)


@pytest.mark.gpu
@pytest.mark.parametrize("mod", ["CoupledModel", "UnCoupledModel"])
def test_split_path_exact_and_across_layouts(mod, tmp_path, monkeypatch):
    """2048^2 on the split transforms with the fused spectral kernels (NIWQG_SPLIT=1), 2 + 2 steps: exact.  A checkpoint
    written on the cluster-kernel path (NIWQG_SPLIT=0) and resumed on the split path agrees with the uninterrupted run."""
    N, n = 2048, 2
    kw, U0, k0 = lamb_params(N, True, 1, 100)
    kw.update(twrite=10 ** 9, tdiags=2)
    cls = _cls(mod)

    def run(split, nsteps, seed_variant=0):
        monkeypatch.setenv("NIWQG_SPLIT", split)
        m = cls(**kw)
        _seed(m, mod, U0, k0, variant=seed_variant)
        for _ in range(nsteps):
            m._step_forward()
        return m

    ref = _snapshot(run("1", 2 * n))
    b = run("1", n)
    b.save_checkpoint(str(tmp_path / "split"))
    dirty = run("1", n + 1, seed_variant=1)
    dirty.load_checkpoint(str(tmp_path / "split"))
    for _ in range(n):
        dirty._step_forward()
    _assert_same(_snapshot(dirty), ref)
    del b, dirty

    ref0 = run("0", 2 * n)
    b0 = run("0", n)
    b0.save_checkpoint(str(tmp_path / "nosplit"))
    del b0
    monkeypatch.setenv("NIWQG_SPLIT", "1")
    c = cls.from_checkpoint(str(tmp_path / "nosplit"))
    for _ in range(n):
        c._step_forward()
    for f in ("q", "qh", "phi", "phih", "u", "v"):
        assert rel_l2(getattr(c, f), getattr(ref0, f)) <= 1e-13, f
    for k in ("Ke", "Pw", "Kw"):
        assert abs(getattr(c, k) - getattr(ref0, k)) <= 1e-13 * abs(getattr(ref0, k)), k
    assert (c.t, c.tc) == (ref0.t, ref0.tc)


@pytest.mark.gpu
@pytest.mark.skipif(not os.environ.get("NIWQG_SLOW_TESTS"), reason="writes a ~9 GiB checkpoint (set NIWQG_SLOW_TESTS=1)")
def test_8192_default_path_restores_bitwise(tmp_path):
    from niwqg_b200 import CoupledModel
    N = 8192
    kw, U0, k0 = lamb_params(N, True, 1, 100)
    kw.update(twrite=10 ** 9, tdiags=10 ** 9)
    m = CoupledModel.Model(**kw)
    m._h.ic("LambDipole", [U0, 2 * np.pi / k0])
    m._h.ic("Uniform", [2 * U0 / np.sqrt(2), 2 * U0 / np.sqrt(2)])
    m._step_forward()
    m.save_checkpoint(str(tmp_path / "ck"))
    m._step_forward()
    x = (m.q, m.phi, m.Ke, m.Pw, m.Kw)
    m.load_checkpoint(str(tmp_path / "ck"))
    m._step_forward()
    y = (m.q, m.phi, m.Ke, m.Pw, m.Kw)
    for a, b in zip(x, y):
        assert np.array_equal(a, b)


@pytest.mark.gpu
def test_mismatches_are_refused_and_leave_the_model_untouched(tmp_path):
    import json
    from niwqg_b200 import CoupledModel, UnCoupledModel
    mod, kw, U0, k0 = _kw("coupled_filt")
    b = CoupledModel.Model(**kw)
    _seed(b, mod, U0, k0)
    b._step_forward()
    path = str(tmp_path / "ck")
    b.save_checkpoint(path)

    def target(cls=CoupledModel.Model, **over):
        m = cls(**dict(kw, **over))
        _seed(m, mod, U0, k0, variant=1, batch=m.batch)
        m._step_forward(); m._step_forward()
        return m

    def refused(m, exc, match, p=path):
        before = _snapshot(m)
        with pytest.raises(exc, match=match):
            m.load_checkpoint(p)
        _assert_same(_snapshot(m), before)

    refused(target(UnCoupledModel.Model), ValueError, "class")
    refused(target(nx=128), ValueError, "nx=64")
    refused(target(batch=2), ValueError, "batch=1")
    refused(target(dt=kw["dt"] * 0.5), ValueError, "dt=")
    m = target()
    meta = json.load(open(os.path.join(path, "checkpoint.json")))
    meta["version"] = 99
    bad = str(tmp_path / "badversion")
    os.makedirs(bad)
    json.dump(meta, open(os.path.join(bad, "checkpoint.json"), "w"))
    refused(m, ValueError, "version", bad)
    os.remove(os.path.join(path, "PHIX.npy"))
    refused(m, FileNotFoundError, "PHIX", path)
    with pytest.warns(UserWarning, match="dt="):
        with pytest.raises(FileNotFoundError):
            CoupledModel.Model.from_checkpoint(path, dt=kw["dt"] * 0.5)


def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
def test_slab_checkpoints_are_exact_and_portable(tmp_path):
    """tools/checkpoint_slab_check.py on 2 ranks: slab save + slab restore exact; a one-GPU checkpoint resumed on 2 ranks
    and a 2-rank checkpoint resumed on one GPU agree with the uninterrupted one-GPU run to 1e-12."""
    if _ngpu() < 2:
        pytest.skip("needs at least 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tools", "checkpoint_slab_check.py"), str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
