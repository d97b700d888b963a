"""Helpers of the parameter-sweep tests (ensembles whose members have their own coefficients)."""
import numpy as np


def phi_plane_wave_factor(kx, ky, N, L, t, f=1e-4, Nb=0.01, m=0.025, U=0., nu4w=0., nuw=0., muw=0.):
    """exp(c t) of the wave equation's linear operator c = -i k U - nu4w |K|^4 - 0.5 i f |K|^2 / kappa^2 - nuw |K|^2 - muw
    (kappa = m f / Nb) at the mode (kx, ky) (indices, ky signed by the FFT convention).  A single plane wave
    phi = A exp(i(k x + l y)) in a flow at rest has uniform |phi|^2 and J(phi*, phi) = 0, so it induces no flow and its
    coefficient evolves by exactly this factor (YBJ and Coupled with q = 0)."""
    k = 2 * np.pi / L * kx
    l = 2 * np.pi / L * (ky if ky < N // 2 else ky - N)
    wv2 = k * k + l * l
    kappa2 = (m * f / Nb) ** 2
    return np.exp((-1j * k * U - nu4w * wv2 * wv2 - 0.5j * f * wv2 / kappa2 - nuw * wv2 - muw) * t)


def phi_plane_wave(kx, ky, N, L, A=1.):
    """A exp(i(k x + l y)) at the cell centres x = (i + 1/2) L / N, and its spectral coefficient at (ky, kx)."""
    x = (np.arange(N) + 0.5) / N * L
    k, l = 2 * np.pi / L * kx, 2 * np.pi / L * ky
    phi = A * np.exp(1j * (k * x[None, :] + l * x[:, None]))
    return phi, A * N * N * np.exp(0.5j * (k + l) * L / N)


def sweep(kw_a, kw_b, keys, defaults):
    """Constructor keywords of a batch of two members: kw_a's, with [a, b] for every key of ``keys`` where they differ
    (``defaults``: the constructor's default of a key that kw_a does not set)."""
    kw = dict(kw_a)
    for k in keys:
        a = kw_a[k] if k in kw_a else defaults[k]
        if k in kw_b and kw_b[k] != a:
            kw[k] = [a, kw_b[k]]
    return kw


def member_kw(kw, b):
    """The keywords of member b of a sweep: every list replaced by its b-th value."""
    return {k: (v[b] if isinstance(v, (list, np.ndarray)) else v) for k, v in kw.items()}
