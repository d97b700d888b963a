"""Development aid: the split transform path (NIWQG_SPLIT=1) against the cluster path (NIWQG_SPLIT=0) on the same model
runs: all four kernel-family models, N = 2048 (or the sizes given as arguments: Coupled only above 2048), a few steps,
field-level comparison."""
import os, sys, logging
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np
logging.disable(logging.CRITICAL)
from niwqg_b200 import CoupledModel, UnCoupledModel, YBJModel, QLModel
from cases import lamb_params, rel_l2

sizes = [int(a) for a in sys.argv[1:]] or [2048]
worst = 0.0
for nx in sizes:
    for name, mod in (("coupled", CoupledModel), ("uncoupled", UnCoupledModel), ("ybj", YBJModel), ("ql", QLModel)):
        if nx > 2048 and name != "coupled":
            continue
        res = {}
        for split in ("0", "1"):
            os.environ["NIWQG_SPLIT"] = split
            kw, U0, k0 = lamb_params(nx, True, 2, 3)
            kw["twrite"] = 10 ** 9
            m = mod.Model(**kw)
            rng = np.random.RandomState(3)
            q = 1e-5 * rng.randn(nx, nx)
            phi = (np.ones((nx, nx)) + 1j) * 0.14 + 0.01 * (rng.randn(nx, nx) + 1j * rng.randn(nx, nx))
            m.set_q(q); m.set_phi(phi)
            for _ in range(3):
                m._step_forward()
            res[split] = dict(q=m.q.copy(), phi=m.phi.copy(), qh=m.qh.copy(), phih=m.phih.copy(), phix=m.phix.copy(),
                              u=m.u.copy(), Ke=m.Ke, Pw=m.Pw, Kw=m.Kw,
                              diag={k: np.array(v["value"]) for k, v in m.diagnostics.items() if len(np.atleast_1d(v["value"]))})
            m._h.close()
            del m
        a, b = res["0"], res["1"]
        errs = {k: rel_l2(b[k], a[k]) for k in ("q", "phi", "qh", "phih", "phix", "u")}
        for k in ("Ke", "Pw", "Kw"):
            errs[k] = abs(a[k] - b[k]) / max(abs(a[k]), 1e-300)
        dmax = 0.0
        for k in a["diag"]:
            x, y = np.atleast_1d(a["diag"][k]).astype(float), np.atleast_1d(b["diag"][k]).astype(float)
            if x.size and x.shape == y.shape:
                dmax = max(dmax, float(np.max(np.abs(x - y)) / max(np.max(np.abs(x)), 1e-300)))
        errs["diag"] = dmax
        worst = max(worst, max(v for k, v in errs.items() if k not in ("Pw", "diag")))
        print("N=%d %-9s " % (nx, name) + " ".join("%s %.1e" % kv for kv in errs.items()), flush=True)
print("worst field error %.2e" % worst)
assert worst < 1e-11
