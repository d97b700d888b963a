"""Step time of a parameter sweep: an ensemble whose members share their ETDRK4 tables against the same ensemble with
one table set per member (a swept coefficient), CUDA-event timed on the handle's stream.

    python tools/sweep_time.py [--steps 20] [--repeats 3] [--out FILE.json]

Cases: Coupled 512^2 x 256 sweeping m (phi tables per member) and U (q and phi tables per member), Coupled 2048^2 x 8
sweeping U, QG 512^2 x 64 sweeping U.  Shared and per-member handles are timed alternately, ``--repeats`` times
each; the spread of the repeats is reported with the median.  The GPU name and power limit are read in the same run.
"""
import argparse
import json
import logging
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

CASES = [("coupled", 512, 256, "m"), ("coupled", 512, 256, "U"), ("coupled", 2048, 8, "U"), ("qg", 512, 64, "U")]


def _model(model, N, B, swept):
    from niwqg_b200 import CoupledModel, QGModel
    L, dt = 2 * np.pi * 200e3, 2000. * 128 / N
    kw = dict(nx=N, L=L, dt=dt, batch=B, twrite=10 ** 9, tdiags=10 ** 9, use_filter=True, U=-0.1)
    s = np.linspace(1.0, 0.5, B)
    if model == "qg":
        kw["nu4"] = 7.5e8 * (128 / N) ** 4
        if swept:
            kw["U"] = list(-0.1 * s)
        m = QGModel.Model(**kw)
    else:
        kw.update(m=2 * np.pi / 280, nu4=5e11 * (128 / N) ** 4)
        if swept == "m":
            kw["m"] = list(kw["m"] * (0.5 + s))
        elif swept == "U":
            kw["U"] = list(-0.1 * s)
        m = CoupledModel.Model(**kw)
    rng = np.random.default_rng(1)
    m.set_q(1e-5 * (rng.random((B, N, N)) - 0.5))
    if model != "qg":
        m.set_phi(0.1 * (1 + 1j) + 0.01 * (rng.random((B, N, N)) - 0.5))
    return m


def _gpu():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # the name is still reported
        out = "unknown (%s)" % e
    return name, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    logging.disable(logging.CRITICAL)
    name, power = _gpu()
    rows = []
    for model, N, B, key in CASES:
        handles = {"shared": _model(model, N, B, None), "per_member": _model(model, N, B, key)}
        pm = handles["per_member"]._h.table_members
        for m in handles.values():
            m.step(args.warmup)
        times = {k: [] for k in handles}
        for _ in range(args.repeats):
            for k, m in handles.items():       # alternate: drift of the clock or of the neighbours hits both alike
                times[k].append(m._h.time_steps(args.steps) / args.steps)
        for m in handles.values():
            m._h.close()
        r = dict(model=model, N=N, batch=B, swept=key, per_member_tables=sorted(pm))
        for k, t in times.items():
            r[k + "_ms_per_step"] = float(np.median(t))
            r[k + "_spread_ms"] = [float(min(t)), float(max(t))]
        r["ratio"] = r["per_member_ms_per_step"] / r["shared_ms_per_step"]
        rows.append(r)
        print("%-8s %5d^2 x %3d  sweep %-2s (tables per member: %-7s)  shared %8.3f ms  per-member %8.3f ms  x%.3f"
              % (model, N, B, key, ",".join(sorted(pm)), r["shared_ms_per_step"], r["per_member_ms_per_step"], r["ratio"]),
              flush=True)
    out = dict(gpu=name, power_limit=power, steps=args.steps, warmup=args.warmup, repeats=args.repeats, cases=rows)
    print(json.dumps(out))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
