"""Cost of Lagrangian particles per step (DESIGN.md section 3.4): Coupled 8192^2 with 0, 2^20 and 2^24 particles (waves
on and off) and Coupled 512^2 x 256 members with 4096 particles per member.

Every configuration is timed with CUDA events on the handle's stream (niwqg_time_steps) over `--steps` steps, after two
untimed steps (they capture the step graphs at 512^2).  The configurations alternate on one model, round after round,
and the median of `--rounds` rounds is reported.  Writes JSON with the device name and power limit read in the same run.

    python tools/particles_time.py [--steps 5] [--rounds 3] [--out profiles/particles_time.json]
"""
import argparse
import json
import logging
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def device_info():
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                                      text=True).splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in out.split(",")]
    except Exception as e:      # the timing is still valid; say why the limit is missing
        info["power_limit"] = "unavailable: %s" % e
    return info


def time_case(N, B, configs, steps, rounds):
    from niwqg_b200 import CoupledModel
    from niwqg_b200 import InitialConditions as ic
    from cases import lamb_params
    kw, U0, k0 = lamb_params(N, True, 10 ** 9, 10)
    kw.update(tmax=1e30, twrite=10 ** 9)
    m = CoupledModel.Model(batch=B, **kw)
    q = ic.LambDipole(m, U=U0, R=2 * np.pi / k0)
    m.set_q(q)
    m.set_phi((np.ones_like(q) + 1j) * (2 * U0) / np.sqrt(2))
    rng = np.random.RandomState(0)
    xy = {P: rng.rand(P, 2) * m.L for P, _ in configs if P}
    ms = {c: [] for c in configs}
    for _ in range(rounds):
        for P, waves in configs:
            m.set_particles(xy[P] if P else None, waves=waves)
            m._h.step(2)
            ms[(P, waves)].append(m._h.time_steps(steps) / steps)
    base = float(np.median(ms[(0, False)]))
    rows = []
    for P, waves in configs:
        t = float(np.median(ms[(P, waves)]))
        row = dict(N=N, batch=B, particles_per_member=P, waves=waves, ms_per_step=t, ms_rounds=ms[(P, waves)],
                   overhead_ms=t - base, overhead_pct=100.0 * (t - base) / base)
        if P:
            # particle-stages per second, and the bytes the gathers deliver (16 or 32 double2 of 16 B per stage)
            ps = 4.0 * P * B
            row["particle_stages_per_s"] = ps / ((t - base) * 1e-3) if t > base else None
            row["gathered_GB_per_step"] = ps * (32 if waves else 16) * 16 / 1e9
        rows.append(row)
        print(json.dumps(row), flush=True)
    del m
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "particles_time.json"))
    a = ap.parse_args()
    logging.disable(logging.CRITICAL)
    res = dict(device_info(), steps=a.steps, rounds=a.rounds, cases=[])
    print(json.dumps(res), flush=True)
    cfg8k = [(0, False)] + [(P, w) for P in (2 ** 20, 2 ** 24) for w in (False, True)]
    res["cases"] += time_case(8192, 1, cfg8k, a.steps, a.rounds)
    res["cases"] += time_case(512, 256, [(0, False), (4096, False), (4096, True)], a.steps, a.rounds)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
