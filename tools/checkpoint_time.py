"""Wall time of save_checkpoint / load_checkpoint of a Coupled model on one GPU (default 8192^2, about 9 GiB on disk).
   python tools/checkpoint_time.py [nx] [directory]
The checkpoint goes to a temporary directory under `directory` (default: the system's temporary directory) and is
removed afterwards.  Prints one JSON line with the GPU name and power limit beside the times."""
import json
import logging
import os
import shutil
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np

logging.disable(logging.CRITICAL)
from niwqg_b200 import CoupledModel
from cases import lamb_params

nx = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
base = sys.argv[2] if len(sys.argv) > 2 else None
kw, U0, k0 = lamb_params(nx, True, 1, 100)
kw.update(twrite=10 ** 9, tdiags=10 ** 9)
m = CoupledModel.Model(**kw)
m._h.ic("LambDipole", [U0, 2 * np.pi / k0])
m._h.ic("Uniform", [2 * U0 / np.sqrt(2), 2 * U0 / np.sqrt(2)])
m._step_forward()
m._h.sync()
tmp = tempfile.mkdtemp(dir=base)
try:
    path = os.path.join(tmp, "ck")
    t0 = time.perf_counter()
    m.save_checkpoint(path)
    t_save = time.perf_counter() - t0
    size = sum(os.path.getsize(os.path.join(path, f)) for f in os.listdir(path))
    t0 = time.perf_counter()
    m.load_checkpoint(path)
    m._h.sync()
    t_load = time.perf_counter() - t0
finally:
    shutil.rmtree(tmp, ignore_errors=True)
try:
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, timeout=60).stdout.strip()
except Exception as e:
    gpu = "unknown (%s)" % e
print(json.dumps(dict(model="coupled", nx=nx, slots=m._h.state_slots(), bytes=size, save_s=round(t_save, 2),
                      load_s=round(t_load, 2), save_GBps=round(size / t_save / 1e9, 2),
                      load_GBps=round(size / t_load / 1e9, 2), gpu=gpu)))
