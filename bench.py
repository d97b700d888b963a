#!/usr/bin/env python
"""bench.py -- headline benchmark of the niwqg ETDRK4 hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

Metric (BASELINE.json): fp64 grid-point-steps/s of the coupled NIW-QG model.
Default workload: CoupledModel, Lamb dipole + uniform NIW, 8192^2, fp64, exponential filter on
(the grid the north-star target is stated on; 34.5 GiB resident on one GPU).  With N > 1 the SAME
8192^2 grid is slab-decomposed over the N GPUs (BASELINE config 4: rows of the physical fields / columns of
the spectra per rank, the distributed-FFT transposes fused into the FFT passes as stores into peer memory
over NVLink): strong scaling, "value" = grid-point-steps/s of the one big grid.  `--mode ensemble` instead
steps one independent member per GPU (BASELINE config 5 style, no data-path collective): weak scaling; at
N > 1 the default run reports it too under "ensemble_weak".  One "step" = one _step_etdrk4.

Keys beyond the base contract: `roofline` (dominant kernels: the launches of the 2-D transforms, live CUDA-event
timing), `step_roofline` (whole step against the algorithmic bytes/point model of SURVEY.md section 8d),
`kernel_breakdown`, `launches_per_step`, `cpu_baseline` (the numpy oracle port timed on this box, N=1 only) and, for
N > 1 slab runs, `parity` (slab vs single GPU at 2048^2 and 8192^2).  Other BASELINE configs: `--workload qg128 |
coupled512 | ybj2048 | ql2048 | coupled512_ens8` (the last with `--mode ensemble` on N GPUs).

`--impl reference` times the reference's CPU implementation of the same path (the numpy oracle port,
bit-identical to the reference; the reference itself is pure Python + numpy) on the host cores.
"""
import argparse
import json
import logging
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np

METRIC = "fp64 grid-point-steps/sec (coupled NIW-QG)"
UNIT = "grid-point-steps/s"
# algorithmic bytes per grid point per step (SURVEY.md section 8d: 64 B per 2-D FFT + compulsory state traffic)
B_ALG = {"coupled": 3392.0, "qg": 856.0, "ybj": 1424.0, "ql": 64.0 * 40 + 1088.0}
B_ALG_COUPLED = B_ALG["coupled"]
FFT_PASS_BYTES_PER_POINT = 32.0   # one pass of a c128 2-D FFT: read 16 B + write 16 B (a 2-D transform = two passes)

WORKLOADS = {
    # name: (model, nx, batch)                      BASELINE.json config
    "coupled8192": ("coupled", 8192, 1),          # 4 (slab-decomposed with --gpus N > 1) and the north-star target grid
    "coupled4096": ("coupled", 4096, 1),
    "coupled2048": ("coupled", 2048, 1),
    "coupled512_ens8": ("coupled", 512, 8),       # 5: 8 members of 512^2 per GPU (64 members on 8 GPUs with --mode ensemble)
    "coupled512": ("coupled", 512, 1),            # 2: Lamb dipole + uniform NIW with the energy-budget diagnostics (e2e leg)
    "qg128": ("qg", 128, 1),                      # 1: examples/LambDipole_qg.py (launch-bound: see launches_per_step)
    "ybj2048": ("ybj", 2048, 1),                  # 3: random-spectrum turbulence
    "ql2048": ("ql", 2048, 1),                    # 3
}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def csrc_hash():
    """Identity of the FFT kernel sources a traffic profile belongs to (profiles/traffic.json carries the hash it was
    captured on): the files that define the 2-D transform launches."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "niwqg_b200", "csrc")
    for f in ("common.cuh", "fft_core.cuh", "fft2d.cuh", "fft_split.cuh"):
        with open(os.path.join(d, f), "rb") as fh:
            h.update(f.encode()); h.update(fh.read())
    return h.hexdigest()[:16]


def workload_params(nx, model="coupled"):
    from cases import lamb_params
    qg = model == "qg"
    kw, U0, k0 = lamb_params(nx, not qg, 10 ** 9, 1, qg=qg)     # examples/LambDipole_qg.py runs without the filter
    kw["tmax"] = 1e30
    kw["twrite"] = 10 ** 9
    return kw, U0, k0


def model_class(model):
    from niwqg_b200 import CoupledModel, QGModel, YBJModel, QLModel
    return {"coupled": CoupledModel, "qg": QGModel, "ybj": YBJModel, "ql": QLModel}[model].Model


def initial_conditions(model, U0, k0, batch, seed0=0):
    """Lamb dipole (+ a member-dependent random-spectrum perturbation for ensembles) and a uniform NIW."""
    from niwqg_b200 import InitialConditions as ic
    q = ic.LambDipole(model, U=U0, R=2 * np.pi / k0)
    if batch > 1:
        rng = np.random.RandomState(1234 + seed0)
        q = np.stack([q * (1.0 + 0.01 * b) + 1e-3 * np.abs(q).max() * rng.randn(*q.shape) for b in range(batch)])
    phi = (np.ones(q.shape) + 1j) * (2 * U0) / np.sqrt(2)
    return q, phi


class ClockSampler(object):
    """nvidia-smi clocks during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, pw, reasons = [], [], [], set()
        for line in self.f.read().strip().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            # under load = samples in the upper half of the power range
            thr = 0.5 * (max(pw) + min(pw)) if pw else 0
            load = [s for s, p in zip(sm, pw) if p >= thr] or sm
            out.update(sm_mhz=float(np.median(load)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                       samples=len(sm), power_w_max=float(max(pw)))
        return out


DUMP_MAX_POINTS = 1 << 21     # q (8 B) + phi (16 B) per point: a dump stays under 48 MB at any grid size


def dump_outputs(out_dir, h, qg, suffix=""):
    """Write what the timed steps computed, as a caller of the stepping path receives it, to out_dir/<name><suffix>.npy:
    the physical fields q and phi of every member (phi as float64 with a last axis of (real, imag)) and the integrated
    budgets Ke, Pw, Kw per member.  Fields of more than DUMP_MAX_POINTS points are sampled at fixed points (seeded, the
    same in every run and build), so two builds run with the same arguments can be compared output for output."""
    from niwqg_b200 import _native as nat
    q = h.field("Q")
    phi = None if qg else h.field("PHI")
    if q.size > DUMP_MAX_POINTS:
        idx = np.unique(np.random.RandomState(0).randint(0, q.size, DUMP_MAX_POINTS))
        q = q.reshape(-1)[idx]
        phi = None if qg else phi.reshape(-1)[idx]
    out = {"q": q}
    if not qg:
        out["phi"] = np.stack([phi.real, phi.imag], axis=-1)
    sc = h.scalars()
    for name, slot in (("Ke", "KE"),) if qg else (("Ke", "KE"), ("Pw", "PW"), ("Kw", "KW")):
        out[name] = sc[:, nat.S[slot]]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def slab_parity(dist, local, rank, world):
    """N > 1: the slab-decomposed run against the single-GPU run of the same model (rank 0 holds both).
    (1) 2048^2, 3 steps from a perturbed Lamb dipole: q, phi, qh, Ke;  (2) 8192^2, 2 steps from the bench initial condition
    generated on the device: rel-L2 of q.  The 2048^2 configuration is the one the CUDA path is checked at against the numpy
    oracle (tests/test_gpu_large.py), so this ties the 8-rank geometry to the reference."""
    from niwqg_b200 import CoupledModel, slab, InitialConditions as ic, _native as nat
    from cases import lamb_params, rel_l2
    out = {}
    nx = 2048
    kw, U0, k0 = lamb_params(nx, True, 10 ** 9, 3)
    kw["twrite"] = 10 ** 9
    ms = slab.make_model(CoupledModel.Model, dist=dist, device=local, **kw)
    ref = CoupledModel.Model(device=local, **kw) if rank == 0 else None
    src = ref if rank == 0 else ms
    q0 = ic.LambDipole(src, U=U0, R=2 * np.pi / k0)
    rng = np.random.RandomState(3)
    q0 = q0 + 0.05 * np.abs(q0).max() * rng.randn(nx, nx)
    phi0 = (np.ones_like(q0) + 1j) * (2 * U0) / np.sqrt(2) * (1 + 0.1 * rng.randn(nx, nx))
    for mdl in (ms, ref):
        if mdl is not None:
            mdl.set_q(q0); mdl.set_phi(phi0)
            mdl.step(3)
    qg, pg = slab.gather_rows(ms, ms.q, dist), slab.gather_rows(ms, ms.phi, dist)
    qhg = slab.gather_columns(ms, ms.qh, dist)
    if rank == 0:
        out.update(nx2048_q=rel_l2(qg, ref.q), nx2048_phi=rel_l2(pg, ref.phi), nx2048_qh=rel_l2(qhg, ref.qh),
                   nx2048_Ke=abs(ms.Ke - ref.Ke) / abs(ref.Ke))
        ref._h.close()
    ms._h.close()
    del ms, ref, q0, phi0, qg, pg, qhg
    nx = 8192
    kw, U0, k0 = lamb_params(nx, True, 10 ** 9, 2)
    kw["twrite"] = 10 ** 9
    ms = slab.make_model(CoupledModel.Model, dist=dist, device=local, **kw)
    ref = CoupledModel.Model(device=local, **kw) if rank == 0 else None
    for mdl in (ms, ref):
        if mdl is not None:
            ic.LambDipole(mdl, U=U0, R=2 * np.pi / k0, on_device=True)
            ic.UniformWave(mdl, phi0=(1 + 1j) * (2 * U0) / np.sqrt(2))
            mdl.step(2)
    qg = slab.gather_rows(ms, ms.q, dist)
    if rank == 0:
        out.update(nx8192_q=rel_l2(qg, ref.q), nx8192_Ke=abs(ms.Ke - ref.Ke) / abs(ref.Ke))
        ref._h.close()
    ms._h.close()
    return out


def run_ours(args):
    logging.disable(logging.CRITICAL)
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        # NCCL prints its version banner on stdout when NCCL_DEBUG=VERSION: keep stdout to the one JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            os.environ.pop("NCCL_DEBUG")
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if dist is not None:
        dist.barrier()
    from niwqg_b200 import CoupledModel, slab, _native as nat, InitialConditions as ic

    model_name, nx, batch = WORKLOADS[args.workload]
    cls = model_class(model_name)
    qg = model_name == "qg"
    slab_mode = world > 1 and args.mode == "slab"
    if slab_mode and (batch != 1 or qg):
        raise SystemExit("slab mode needs a single-member kernel-family workload")
    kw, U0, k0 = workload_params(nx, model_name)
    kw_e2e = dict(kw)
    kw_e2e["tdiags"] = 1
    if slab_mode:
        m = slab.make_model(cls, dist=dist, device=local, **kw_e2e)
        q, phi = initial_conditions(m, U0, k0, batch, seed0=0)
        lo, hi = slab.rows_of(rank, world, nx)
        q, phi = np.ascontiguousarray(q[lo:hi]), np.ascontiguousarray(phi[lo:hi])
    else:
        m = cls(batch=batch, device=local, **kw_e2e)
        if model_name in ("ybj", "ql"):
            # BASELINE config 3: random red spectrum (McWilliams 1984), generated on the device, fixed Philox seed
            ic.McWilliams1984(m, k0=k0, E=U0 ** 2 / 2, on_device=True, seed=7 + rank)
            q = m.q
            phi = (np.ones(q.shape) + 1j) * (2 * U0) / np.sqrt(2)
        else:
            q, phi = initial_conditions(m, U0, k0, batch, seed0=rank)
    nyl = nx // world if slab_mode else nx
    # pinned host buffers (torch is used for pinned/host plumbing and the process group only)
    q_pin = torch.empty(q.shape, dtype=torch.float64).pin_memory()
    q_pin.numpy()[...] = q
    qo_pin = torch.empty((batch, nyl, nx), dtype=torch.float64).pin_memory()
    if not qg:
        phi_pin = torch.empty(phi.shape, dtype=torch.complex128).pin_memory()
        phi_pin.numpy()[...] = phi
        po_pin = torch.empty((batch, nyl, nx), dtype=torch.complex128).pin_memory()
    del q, phi
    m.set_q(q_pin.numpy())
    if not qg:
        m.set_phi(phi_pin.numpy())
    h = m._h
    npts = batch * nyl * nx          # grid points this rank steps

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        h.sync()                  # main stream and copy stream: every queued download has landed

    # ---------------- device-resident throughput: K steps, inputs already in HBM
    h.step(args.warmup)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = h.launch_count()
    ms = h.time_steps(args.steps)
    l1 = h.launch_count()
    barrier()
    clk = clocks.stop() if rank == 0 else None
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * npts * args.steps / (ms * 1e-3)     # slab: world * (nx^2 / world) = the one grid
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, h, qg, "_rank%d" % rank if world > 1 else "")

    # ---------------- per-kernel-kind timing (separate short run with events around every launch)
    nprof = min(args.steps, 3)
    h.profile(True)
    h.step(nprof)
    prof = h.profile(False)

    # ---------------- end to end through the public Python API, host buffers both ways
    def stage_next():                          # this step's inputs start their H2D copy while the previous step computes
        if qg:
            m.stage_inputs(q=q_pin.numpy())
        else:
            m.stage_inputs(q=q_pin.numpy(), phi=phi_pin.numpy())

    def e2e_step():
        m.set_q()                              # staged H2D (waits for it) + inversion (Kernel.set_q)
        if not qg:
            m.set_phi()                        # staged H2D (Kernel.set_phi)
        stage_next()                           # the NEXT step's inputs: host -> device on the copy stream, asynchronous
        m._step_forward()                      # step + diagnostics tick (scalars D2H) + status
        for b in range(batch):                 # snapshot of the result (every member), D2H: queued on the copy stream, so
            h.field_into("Q", qo_pin.numpy()[b], b, wait=False)         # it overlaps the next step's uploads (full duplex)
            if not qg:
                h.field_into("PHI", po_pin.numpy()[b], b, wait=False)
    stage_next()
    for _ in range(2):
        e2e_step()
    barrier()
    ne = max(2, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(ne):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_val = world * npts * ne / e2e_s
    h2d = npts * 8 + (0 if qg else npts * 16)
    d2h = npts * (8 if qg else 24) + nat.S_COUNT * 8 * batch
    diag_ke = m.diagnostics["ke_qg"]["value"]

    ens = None
    if slab_mode and not args.no_ensemble:
        # the other natural partition of the north star: one independent member per GPU, no collective (weak scaling)
        h.close()
        del m, h
        me = cls(batch=1, device=local, **kw)
        qe, pe = initial_conditions(me, U0, k0, 1, seed0=rank)
        me.set_q(qe); me.set_phi(pe)
        del qe, pe
        me._h.step(args.warmup)
        barrier_e = lambda: (dist.barrier(), torch.cuda.synchronize(), me._h.sync())
        barrier_e()
        ms_e = me._h.time_steps(args.steps)
        barrier_e()
        t = torch.tensor([ms_e], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ens = {"value": world * nx * nx * args.steps / (float(t.item()) * 1e-3), "unit": UNIT, "scaling": "weak",
               "ms_per_step": float(t.item()) / args.steps,
               "what": "one independent %d^2 member per GPU, no data-path collective" % nx}
        me._h.close()
        del me
    parity = None
    if slab_mode and not args.no_check:
        try:
            h.close()
        except Exception:
            pass
        parity = slab_parity(dist, local, rank, world)
    ens512 = None
    if world == 1 and not args.no_ensemble and args.workload == "coupled8192":
        # BASELINE config 5 on one GPU: an ensemble of independent 512^2 members batched through the same kernels
        # (every FFT pass fits one tile: no cluster exchange)
        h.close()
        del m, h
        nb, ne_ = 256, 512
        kw5, U5, k5 = workload_params(ne_)
        m5 = CoupledModel.Model(batch=nb, device=local, **kw5)
        q5, p5 = initial_conditions(m5, U5, k5, nb, seed0=0)
        m5.set_q(q5); m5.set_phi(p5)
        del q5, p5
        m5._h.step(3)
        m5._h.sync()
        ms5 = m5._h.time_steps(3) / 3
        v5 = nb * ne_ * ne_ / (ms5 * 1e-3)
        ens512 = {"value": v5, "unit": UNIT, "ms_per_step": ms5, "members": nb, "nx": ne_,
                  "step_roofline_frac": B_ALG_COUPLED * v5 / 1e9 / measured_peaks()[0],
                  "what": "256 independent CoupledModel 512^2 members (1 GiB per field) stepped as one batch on one GPU"}
        m5._h.close()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    peak, peak_src = measured_peaks()
    # dominant kernels = the launches of the 2-D transforms: row passes, column passes and - where a grid's lines do not
    # fit one tile - the streaming radix stage ("fft_p"; zero when it is fused into the spectral kernels).  A 2-D transform
    # is two passes of 32 B per point whatever the number of launches it takes.
    # "fft_row_ld" / "fft_row_ld2" = forward row passes that form their input from three / two physical fields while
    # loading them (the wave-PV pair: reads 48 B; (uq, vq): reads 32 B; both write 16 B per point) - 32 / 16 B per point
    # more than a plain pass, and no pointwise kernel (or no store + re-read of the product).
    fft_kinds = ("fft_row", "fft_col", "fft_p", "fft_row_ld", "fft_row_ld2")
    fft_ms = sum(prof[k][0] for k in fft_kinds)
    n_ld, n_ld2 = prof["fft_row_ld"][1], prof["fft_row_ld2"][1]
    n2d = max(prof["fft_row"][1] + n_ld + n_ld2, prof["fft_col"][1])   # 2-D transforms in the profiled steps
    total_prof = sum(v[0] for v in prof.values())
    pass_bytes = FFT_PASS_BYTES_PER_POINT * npts
    achieved = (2 * n2d + n_ld + 0.5 * n_ld2) * pass_bytes / (fft_ms * 1e-3) / 1e9 if fft_ms > 0 else 0.0
    traffic, traffic_note = None, "no ncu capture on record for this workload"
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        rec = tj.get(args.workload)
        if isinstance(rec, dict):
            if rec.get("csrc_hash") == csrc_hash():
                traffic, traffic_note = rec["dram_bytes_per_pass"], rec.get("source", "")
            else:
                traffic_note = "ncu capture on record is of other kernel sources (csrc hash %s, now %s)" % (rec.get("csrc_hash"), csrc_hash())
    except Exception:
        pass
    b_alg = B_ALG[model_name]
    big = nx * nyl * batch * 16 * 30 > 4e8
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak" if (world > 1 and not slab_mode) else "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s %s %d^2 fp64, %s, %d member(s)/GPU (%s)"
                               % ({"coupled": "CoupledModel", "qg": "QGModel", "ybj": "YBJModel", "ql": "QLModel (repaired)"}[model_name],
                                  "random-spectrum turbulence (McWilliams 1984) + uniform NIW" if model_name in ("ybj", "ql")
                                  else ("Lamb dipole" if qg else "Lamb dipole + uniform NIW"),
                                  nx, "no filter (examples/LambDipole_qg.py)" if qg else "exponential filter", batch, args.workload),
                   "parallelism": ("slab decomposition of the one grid over %d GPUs: rows/columns per rank, FFT transposes "
                                   "fused into the FFT passes as peer-memory stores over NVLink (%s), all-reduced budget sums"
                                   % (world, "CUDA IPC" if os.environ.get("NIWQG_SLAB_NCCL", "0") != "1" else "NCCL all-to-all"))
                                  if slab_mode else
                                  ("ensemble: one member batch per GPU, no data-path collective" if world > 1 else "single GPU"),
                   "l2": "working set %.1f GiB per GPU >> 126 MB L2 (inputs larger than L2, no flush needed)"
                         % (batch * nyl * nx * 16 * 34.5 / 2 ** 30) if big else
                         "working set fits in L2: not an HBM-bound measurement (launch-bound: see launches_per_step)"},
        "clocks": clk,
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": ne, "what": "per step: set_q%s from pinned host arrays (double-buffered input pipeline: the host-to-device copy of "
                                     "step i+1's arrays is queued with stage_inputs() before step i runs and overlaps it), _step_forward() with the "
                                     "diagnostics tick (scalars to host), q%s of every member copied back to pinned host arrays (asynchronous "
                                     "downloads: they overlap the next step; all have landed when the clock stops)"
                                     % (("", "") if qg else (" + set_phi", " and phi"))},
        "gpu_launches": int(l1 - l0),
        "launches_per_step": (l1 - l0) / float(args.steps),
        "us_per_step": 1e3 * ms / args.steps,
        "roofline": {"bound": "hbm", "kernel": "2-D FFT launches (k_fft_pass row passes, k_fft_colsub2 / k_fft_pass column passes"
                                               ", k_split_p radix stage)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "traffic_note": traffic_note, "peak_source": peak_src, "bytes_per_launch": pass_bytes,
                     "avg_launch_ms": fft_ms / max(sum(prof[k][1] for k in fft_kinds), 1), "transforms_per_step": n2d / float(nprof),
                     "row_pass_gbs": pass_bytes / (prof["fft_row"][0] / max(prof["fft_row"][1], 1) * 1e-3) / 1e9,
                     "col_pass_gbs": pass_bytes / ((prof["fft_col"][0] + prof["fft_p"][0]) / max(prof["fft_col"][1], 1) * 1e-3) / 1e9,
                     "share_of_step": fft_ms / total_prof,
                     "loader_row_passes_per_step": (n_ld + n_ld2) / float(nprof),
                     "what": "achieved = 64 B per point per 2-D transform (+ 32 / 16 B per point for a row pass that forms its input from "
                             "three / two fields while loading them) / time of ALL transform launches (live CUDA events)"},
        "step_roofline": {"bytes_per_point_step": b_alg, "achieved": b_alg * value / world / 1e9,
                          "peak": peak, "unit": "GB/s", "frac": b_alg * value / world / 1e9 / peak},
        "kernel_breakdown": {k: {"ms_per_step": v[0] / nprof, "launches_per_step": v[1] / nprof} for k, v in prof.items()},
        "sanity": {"ke_qg_last": float(np.ravel(diag_ke)[-1]), "finite": bool(np.all(np.isfinite(diag_ke)))},
    }
    if parity is not None:
        out["parity"] = parity
    if ens is not None:
        out["ensemble_weak"] = ens
    if ens512 is not None:
        out["ensemble_512x256_one_gpu"] = ens512
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(budget_s=25.0)
    print(json.dumps(out), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def _oracle_model(nx, model="coupled"):
    from oracle import niwqg_oracle as orc
    kw, U0, k0 = workload_params(nx, model)
    kw.pop("tdiags", None)
    if model == "qg":
        o = orc.QGOracle(tdiags=10 ** 9, **kw)
        o.set_q(orc.lamb_dipole(o, U=U0, R=2 * np.pi / k0))
        return o
    o = orc.NIWQGOracle(model=model, tdiags=10 ** 9, **kw)
    if model in ("ybj", "ql"):
        np.random.seed(7)
        q = orc.mcwilliams1984(o, k0=k0, E=U0 ** 2 / 2)
    else:
        q = orc.lamb_dipole(o, U=U0, R=2 * np.pi / k0)
    o.set_q(q)
    o.set_phi((np.ones_like(q) + 1j) * (2 * U0) / np.sqrt(2))
    return o


def cpu_baseline(budget_s=25.0, nx=None, steps=None):
    """The numpy oracle port (bit-identical to the reference) timed on this box, one core (numpy's FFT and
    ufuncs are single-threaded).  Bounded sample of the same workload: same model, parameters scaled the same
    way, smaller grid - the metric is per grid point."""
    if nx is None:
        nx = 1024 if budget_s >= 20 else 512
    per_step = {256: 0.3, 512: 1.3, 1024: 6.5}.get(nx, 6.5)
    if steps is None:
        steps = max(2, int(budget_s / per_step))
    o = _oracle_model(nx)
    o.step()                                   # warm-up
    t0 = time.perf_counter()
    for _ in range(steps):
        o.step()
    dt = time.perf_counter() - t0
    return {"value": nx * nx * steps / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "host_cores_available": os.cpu_count(),
            "sample": "CoupledModel Lamb dipole + uniform NIW %d^2 (same parameters scaled to the grid), %d steps of "
                      "oracle/niwqg_oracle.py (numpy, bit-identical to the reference), %.1f s" % (nx, steps, dt)}


def _ref_worker(nx, steps, warm, q, model="coupled"):
    o = _oracle_model(nx, model)
    for _ in range(warm):
        o.step()
    t0 = time.perf_counter()
    for _ in range(steps):
        o.step()
    q.put(time.perf_counter() - t0)


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path (numpy; oracle port), using all the host
    threads it can: the solver itself is single-threaded, so the box's cores are used the only way the
    reference can use them - independent single-threaded replicas (an ensemble) run concurrently."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    total_steps = args.steps + args.warmup
    model_name, nx_w, batch = WORKLOADS[args.workload]
    # bounded sample: keep the whole run within a few minutes (per-step costs of the coupled model; the others are cheaper)
    nx = 1024 if total_steps * 6.5 <= 150 else (512 if total_steps * 1.3 <= 150 else 256)
    nx = min(nx, nx_w)
    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        pass
    mem_per = {256: 0.3, 512: 1.2, 1024: 4.5}.get(nx, 0.3) * 2 ** 30
    try:
        avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    except Exception:
        avail = 8 * 2 ** 30
    nproc = int(max(1, min(cores, 32, avail * 0.6 // mem_per)))
    ctx = mp.get_context("fork")
    qq = ctx.Queue()
    procs = [ctx.Process(target=_ref_worker, args=(nx, args.steps, args.warmup, qq, model_name)) for _ in range(nproc)]
    for p in procs:
        p.start()
    times = [qq.get() for _ in procs]
    for p in procs:
        p.join()
    wall = max(times)
    value = nproc * nx * nx * args.steps / wall
    sample = ("%d concurrent single-threaded replicas of the %s model of this workload at %d^2, %d steps each "
              "(oracle/niwqg_oracle.py = the reference's numpy arithmetic), %.1f s" % (nproc, model_name, nx, args.steps, wall))
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": "%s model %d^2 fp64 (%s); CPU arm times a bounded %d^2 sample"
                                  % (model_name, nx_w, args.workload, nx)},
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": nproc, "kind": "port", "sample": sample,
                            "single_replica_value": nx * nx * args.steps / float(np.mean(times))},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="coupled8192", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--mode", default="slab", choices=["slab", "ensemble"],
                    help="N > 1: slab-decompose the one grid (strong scaling, default) or one member per GPU (weak)")
    ap.add_argument("--no-ensemble", action="store_true", help="N > 1 slab run: skip the extra ensemble_weak measurement")
    ap.add_argument("--no-check", action="store_true", help="N > 1 slab run: skip the parity leg (slab vs single GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write q, phi (a fixed sample of points on large grids) and the budgets "
                         "Ke, Pw, Kw as DIR/<name>.npy (float64; _rank<r> appended with N > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
