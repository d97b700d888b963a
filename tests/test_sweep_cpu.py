"""CPU checks of parameter sweeps (ensemble members with their own coefficients): the ABI struct, keyword validation,
checkpoint keywords as lists, and the wave plane-wave factor the GPU tests use."""
import logging
import os
import re

import numpy as np
import pytest

from sweep_cases import member_kw, phi_plane_wave, phi_plane_wave_factor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
logging.disable(logging.CRITICAL)


def _header_struct_fields(name):
    header = open(os.path.join(ROOT, "include", "niwqg_b200.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), header, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in body.split(";"):
        decl = " ".join(decl.split())
        if not decl:
            continue
        m = re.match(r"(size_t|int|double|char)\s+(.*)", decl)
        assert m, decl
        fields += [(n.strip(), m.group(1)) for n in m.group(2).split(",")]
    return fields


def test_member_params_struct_matches_header_and_native():
    """The ctypes mirror of niwqg_member_params lists exactly the header's fields, in order, and every coefficient it
    holds is a field of niwqg_params of the same name (members replace those fields of p)."""
    import ctypes as C
    from niwqg_b200 import _native
    want = _header_struct_fields("niwqg_member_params")
    assert want[0] == ("struct_size", "size_t")
    names = {C.c_size_t: "size_t", C.c_int: "int", C.c_double: "double"}
    assert [(n, names[t]) for n, t in _native.MemberParams._fields_] == want
    params = dict(_header_struct_fields("niwqg_params"))
    for n, t in want[1:]:
        assert params.get(n) == "double", n
    assert tuple(n for n, _ in want[1:]) == _native.MEMBER_KEYS
    for eq, keys in _native.TABLE_KEYS.items():
        assert set(keys) <= set(_native.MEMBER_KEYS), eq


def test_member_keywords_validation():
    from niwqg_b200 import _native as nat
    kw = nat.member_keywords(3, dict(U=0.1, f=[1e-4, 2e-4, 3e-4]), dict(nx=64, L=1e6))
    assert kw["U"] == 0.1 and kw["f"].dtype == np.float64 and kw["f"].shape == (3,)
    with pytest.raises(ValueError, match="f"):
        nat.member_keywords(3, dict(f=[1e-4, 2e-4]), {})
    with pytest.raises(ValueError, match="nu4w"):
        nat.member_keywords(2, dict(nu4w=[[0., 1.]]), {})
    for k in ("dt", "L", "use_filter"):
        with pytest.raises(ValueError, match=k):
            nat.member_keywords(2, {}, {k: [1., 2.]})


def test_checkpoint_keywords_round_trip_as_lists(tmp_path):
    """Per-member keywords (arrays on the model) are written as lists and compare element-wise on load: equal lists
    match, a different list, a list against a scalar and a scalar against a list do not, and the error names the
    keyword."""
    from niwqg_b200 import Checkpoint

    class Model(object):
        _checkpoint_attr = {}
        _checkpoint_params = ("dt", "U", "nu4w")

    m = Model()
    m.dt, m.U, m.nu4w = 100., np.array([0.1, -0.2]), np.float64(0.)
    kw = Checkpoint._keywords(m, m._checkpoint_params)
    assert kw == {"dt": 100., "U": [0.1, -0.2], "nu4w": 0.}
    assert isinstance(kw["U"], list)

    class IO(object):
        nx, batch, rank, nranks = 8, 2, 0, 1

        def slots(self):
            return [Checkpoint.Slot("QH", np.complex128, (8, 8), "cols")]

        def read(self, name, member):
            return np.full((8, 8), member + 1j)

        def get_carry(self):
            return np.arange(4.)

        def agree(self, ok):
            return ok

    path = str(tmp_path / "ck")
    Checkpoint.write(path, dict(model="x", params=kw, run={}, t=0., tc=0, status={}), IO())
    meta = Checkpoint.read_meta(path)
    assert meta["params"]["U"] == [0.1, -0.2] and meta["params"]["nu4w"] == 0.
    same = Checkpoint._same
    assert same(np.array([0.1, -0.2]), meta["params"]["U"])
    assert not same(np.array([0.1, -0.3]), meta["params"]["U"])
    assert not same(0.1, meta["params"]["U"]) and not same([0., 0.], meta["params"]["nu4w"])
    assert same(100., meta["params"]["dt"]) and not same(None, 1.)
    assert member_kw(dict(meta["params"]), 1) == {"dt": 100., "U": -0.2, "nu4w": 0.}


@pytest.mark.parametrize("model", ["ybj", "coupled"])
def test_phi_plane_wave_factor_matches_oracle(model):
    """A plane wave phi in a flow at rest (q = 0) evolves by exactly phi_plane_wave_factor in the numpy oracle, with
    every coefficient of the wave operator non-zero (the formula the per-member GPU tests use)."""
    from oracle import niwqg_oracle as orc
    N, L, dt, nsteps, A = 32, 5e5, 2000., 4, 1e-6
    kx, ky = 5, N - 3
    T = nsteps * dt
    wv2 = (2 * np.pi / L) ** 2 * (kx * kx + 9)
    kw = dict(nx=N, L=L, dt=dt, use_filter=False, f=1.2e-4, N=0.008, m=0.03, U=0.3 / (2 * np.pi / L * kx * T),
              nu4=0., nu=0., mu=0., nu4w=0.4 / (wv2 * wv2 * T), nuw=0.3 / (wv2 * T), muw=0.2 / T,
              twrite=10 ** 9, tdiags=10 ** 9, tmax=T - 1.)
    o = orc.NIWQGOracle(model=model, **kw)
    phi, c0 = phi_plane_wave(kx, ky - N, N, L, A)
    o.set_q(np.zeros((N, N)))
    o.set_phi(phi)
    for _ in range(nsteps):
        o.step_forward()
    want = c0 * phi_plane_wave_factor(kx, ky, N, L, T, f=kw["f"], Nb=kw["N"], m=kw["m"], U=kw["U"], nu4w=kw["nu4w"],
                                      nuw=kw["nuw"], muw=kw["muw"])
    ph = np.fft.fft2(o.phi)
    assert abs(ph[ky, kx] - want) <= 1e-10 * abs(want), (ph[ky, kx], want)
    assert 0.2 < abs(want / c0) < 0.6          # the operator acted
    ph[ky, kx] = 0
    assert np.abs(ph).max() <= 1e-9 * abs(want)
