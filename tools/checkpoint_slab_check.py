"""torchrun target: checkpoints of a slab-decomposed Coupled 256^2 run on WORLD_SIZE GPUs.
   python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 \
       tools/checkpoint_slab_check.py DIR
- slab save -> slab restore into a dirty slab model: bit-for-bit the uninterrupted slab run;
- one-GPU checkpoint resumed on the slab, slab checkpoint resumed on one GPU: both agree with the uninterrupted one-GPU
  run to 1e-12 (rel-L2 of q, phi, qh; relative Ke, Pw, Kw)."""
import functools
import logging
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np
import torch
import torch.distributed as dist

logging.disable(logging.CRITICAL)
from niwqg_b200 import CoupledModel, slab
from niwqg_b200 import InitialConditions as ic
from cases import lamb_params, rel_l2

out_dir = sys.argv[1]
nx, n = 256, 3
cls = CoupledModel.Model
local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
rank, world = dist.get_rank(), dist.get_world_size()
kw, U0, k0 = lamb_params(nx, True, 1, 100)
kw.update(twrite=10 ** 9, tdiags=2)
lo, hi = slab.rows_of(rank, world, nx)


def seed(m, variant=0):
    rng = np.random.RandomState(3 + variant)
    q0 = ic.LambDipole(m, U=U0, R=2 * np.pi / k0)
    m.set_q(q0 * (1 + 0.3 * variant) + 0.05 * np.abs(q0).max() * rng.randn(nx, nx))
    m.set_phi((np.ones((nx, nx)) + 1j) * (2 * U0) / np.sqrt(2) * (1 + 0.1 * rng.randn(nx, nx)))


def steps(m, k):
    for _ in range(k):
        m._step_forward()
    return m


def compare(m, ref, exact):
    """Worst disagreement of slab or one-GPU model m with one-GPU model ref (0.0 required when exact)."""
    part = (lambda a: a[lo:hi]) if m.nranks > 1 else (lambda a: a)
    errs = [rel_l2(m.q, part(ref.q)), rel_l2(m.phi, part(ref.phi)), rel_l2(slab.gather_columns(m, m.qh, dist), ref.qh)]
    errs += [abs(getattr(m, k) - getattr(ref, k)) / abs(getattr(ref, k)) for k in ("Ke", "Pw", "Kw")]
    errs += [float(m.t != ref.t or m.tc != ref.tc)]
    if exact:
        same = all(np.array_equal(np.asarray(m.diagnostics[k]["value"]), np.asarray(ref.diagnostics[k]["value"]))
                   for k in m.diagnostics)
        errs.append(0.0 if same else 1.0)
    return max(errs)


# uninterrupted runs: slab and one GPU (every rank steps its own one-GPU copy)
ref = cls(device=local, **kw)
seed(ref)
steps(ref, 2 * n)
a = slab.make_model(cls, dist=dist, **kw)
seed(a)
steps(a, n)
a.save_checkpoint(os.path.join(out_dir, "slab"), dist)
steps(a, n)

# 1) slab -> slab, into a dirty slab model
d = slab.make_model(cls, dist=dist, **kw)
seed(d, 1)
steps(d, n + 1)
d.load_checkpoint(os.path.join(out_dir, "slab"), dist)
steps(d, n)
e1 = max(rel_l2(d.q, a.q), rel_l2(d.phi, a.phi), rel_l2(d.qh, a.qh), float(d.t != a.t))
e1 = max(e1, *[abs(getattr(d, k) - getattr(a, k)) for k in ("Ke", "Pw", "Kw")])
e1 = max(e1, float(not all(np.array_equal(np.asarray(d.diagnostics[k]["value"]), np.asarray(a.diagnostics[k]["value"]))
                           for k in d.diagnostics)))
# every state slot (this rank's rows / columns) and the scalar carry, bit for bit
e1 = max(e1, float(d._h.state_slots() != a._h.state_slots()))
e1 = max(e1, float(not all(np.array_equal(d._h.field(s, 0), a._h.field(s, 0)) for s in a._h.state_slots())))
e1 = max(e1, float(not np.array_equal(d._h.carry(), a._h.carry())))

# 2) one GPU -> slab
if rank == 0:
    s = cls(device=local, **kw)
    seed(s)
    steps(s, n)
    s.save_checkpoint(os.path.join(out_dir, "single"))
dist.barrier()
r = slab.make_model(functools.partial(cls.from_checkpoint, os.path.join(out_dir, "single")), dist=dist)
steps(r, n)
e2 = compare(r, ref, False)

# 3) slab -> one GPU
g = cls.from_checkpoint(os.path.join(out_dir, "slab"), device=local)
steps(g, n)
e3 = compare(g, ref, False)

print("rank %d/%d coupled %d^2: slab->slab %.1e (exact required), single->slab %.2e, slab->single %.2e"
      % (rank, world, nx, e1, e2, e3), flush=True)
ok = e1 == 0.0 and e2 <= 1e-12 and e3 <= 1e-12
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 1)
