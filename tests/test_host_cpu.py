"""CPU-side checks of the host logic: the FFT engine's index maps replayed on the CPU (including the
thread-block-cluster decimation split), and that the C-ABI library loads and exports every symbol that
include/niwqg_b200.h declares.  No compute calls: there is no GPU in the build container."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_fft_index_maps_on_cpu(tmp_path):
    exe = str(tmp_path / "host_fft_emul")
    subprocess.check_call([NVCC, "-O1", "-Wno-deprecated-gpu-targets", "-o", exe,
                           os.path.join(ROOT, "tests", "host", "host_fft_emul.cu")])
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "C=8" in out.stdout and "N= 8192" in out.stdout


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_fused_kernel_work_unit_geometry_on_cpu(tmp_path):
    """kernels_fused.cuh: every spectral element is owned by exactly one thread of one work unit, lanes l / l+16 hold the
    columns kx / kx+N/2, and the thread named as the holder of -K holds exactly (-ky, -kx) (tests/host/host_fused_map.cu)."""
    import nvidia.nccl as n
    inc = os.path.join(list(n.__path__)[0], "include")
    exe = str(tmp_path / "host_fused_map")
    subprocess.check_call([NVCC, "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-I", inc, "-o", exe,
                           os.path.join(ROOT, "tests", "host", "host_fused_map.cu")])
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.count(" 0 mapping errors, 0 elements not owned exactly once") == 3, out.stdout


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as ge
    ge.build()
    from niwqg_b200 import _native
    lib = _native.load()
    header = open(os.path.join(ROOT, "include", "niwqg_b200.h")).read()
    declared = set(re.findall(r"\b(niwqg_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 15
    for name in sorted(declared):
        assert hasattr(lib, name), "libniwqg_b200.so does not export %s" % name
    assert declared == set(_native.EXPORTS), declared ^ set(_native.EXPORTS)


def test_no_cpu_fallback_without_device():
    """The product path must fail loudly when there is no CUDA device (no oracle / numpy fallback)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import logging
    logging.disable(logging.CRITICAL)
    from niwqg_b200 import CoupledModel
    with pytest.raises(RuntimeError):
        CoupledModel.Model(nx=64)


def test_product_path_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "niwqg_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+\S*oracle", src, re.M), "%s imports the oracle" % f
                assert "niwqg_oracle" not in src, "%s references the oracle module" % f


def test_library_reads_no_tuning_switches_from_the_environment():
    """The CUDA library chooses its algorithms from the problem (model, grid, batch, ranks), not from environment switches:
    it reads NIWQG_SPLIT (the tests select the cluster-kernel reference path with it) and NIWQG_NCCL_LIB (where NCCL is).
    NIWQG_SLAB_EXCHANGE and NIWQG_SLAB_BARRIER (copy-engine exchange, all-reduce barrier of slab runs) stay until their
    removal has been checked on several GPUs."""
    names = set()
    for dirpath, _, files in os.walk(os.path.join(ROOT, "niwqg_b200", "csrc")):
        for f in files:
            src = open(os.path.join(dirpath, f)).read()
            for arg in re.findall(r"getenv\s*\(([^)]*)\)", src):
                m = re.fullmatch(r'\s*"(\w+)"\s*', arg)
                assert m, "%s: getenv of a name that is not a literal: %s" % (f, arg)
                names.add(m.group(1))
    assert names == {"NIWQG_SPLIT", "NIWQG_NCCL_LIB", "NIWQG_SLAB_EXCHANGE", "NIWQG_SLAB_BARRIER"}, names


def test_initial_conditions_match_reference_golden():
    """niwqg_b200.InitialConditions (host numpy, vectorised) reproduces the reference generators bit for bit:
    LambDipole against the q0 the unmodified reference produced (tests/golden/make_golden.py), the plane-wave /
    wave-packet formulas against their definitions (niwqg/InitialConditions.py:117-169)."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    from cases import lamb_params, load_golden
    from niwqg_b200 import InitialConditions as ic

    class Grid(object):
        pass
    for nx, name, qg in ((64, "coupled_lamb64_filt", False), (64, "qg_lamb64_filt", True)):
        kw, U0, k0 = lamb_params(nx, True, 2, 10, qg=qg)
        m = Grid()
        m.nx = nx
        m.x, m.y = np.meshgrid(np.arange(0.5, nx, 1.) / nx * kw["L"], np.arange(0.5, nx, 1.) / nx * kw["L"])
        assert np.array_equal(ic.LambDipole(m, U=U0, R=2 * np.pi / k0), load_golden(name)["q0"])
    k, l = 3e-5, 1e-5
    assert np.array_equal(ic.PlaneWave(m, k=k, l=l, phase=0.3), np.exp(1j * (k * m.x + l * m.y) + 0.3))
    wp = ic.WavePacket(m, k=k, l=l, R=1e5, x0=2e5, y0=1e5)
    r = np.sqrt((m.x - 2e5) ** 2 + (m.y - 1e5) ** 2)
    assert np.allclose(wp, np.exp(1j * (k * (m.x - 2e5) + l * (m.y - 1e5))) * np.exp(-(r / 1e5) ** 2), rtol=1e-15, atol=0)


def _header_params_fields():
    """(name, ctype-string, array-length) of every field of struct niwqg_params, in declaration order."""
    header = open(os.path.join(ROOT, "include", "niwqg_b200.h")).read()
    body = re.search(r"typedef struct niwqg_params \{(.*?)\} niwqg_params;", header, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in body.split(";"):
        decl = " ".join(decl.split())
        if not decl:
            continue
        m = re.match(r"(size_t|int|double|char)\s+(.*)", decl)
        assert m, decl
        for name in m.group(2).split(","):
            name = name.strip()
            arr = re.match(r"(\w+)\[(\d+)\]", name)
            fields.append((arr.group(1), m.group(1), int(arr.group(2))) if arr else (name, m.group(1), 0))
    return fields


def _ctypes_fields(cls):
    import ctypes as C
    names = {C.c_size_t: "size_t", C.c_int: "int", C.c_double: "double"}
    out = []
    for name, tp in cls._fields_:
        if hasattr(tp, "_length_"):
            out.append((name, "char", tp._length_))
        else:
            out.append((name, names[tp], 0))
    return out


def test_params_struct_matches_header_in_native_and_in_integration_doc():
    """The ctypes mirror of niwqg_params (niwqg_b200/_native.py) and the binding INTEGRATION.md tells a reference maintainer
    to add must list exactly the fields of include/niwqg_b200.h, in order - a shorter struct would be over-read by
    niwqg_create (which now also checks struct_size)."""
    import ctypes as C
    want = _header_params_fields()
    assert want[0] == ("struct_size", "size_t", 0) and want[-1] == ("nccl_id", "char", 128) and len(want) >= 27
    from niwqg_b200 import _native
    assert _ctypes_fields(_native.Params) == want
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    snippet = re.search(r"```python\n(import ctypes as C.*?)```", doc, re.S).group(1)
    cls_src = snippet[snippet.index("class Params"):]
    cls_src = cls_src[:re.search(r"\n\S", cls_src[1:]).start() + 1]       # up to the next top-level statement
    ns = {"C": C}
    exec(cls_src, ns)
    assert _ctypes_fields(ns["Params"]) == want
    assert C.sizeof(ns["Params"]) == C.sizeof(_native.Params)


def test_traffic_record_matches_its_capture():
    """profiles/traffic.json (what bench.py reports as roofline.traffic) is reproducible from the committed ncu capture:
    DRAM bytes of all transform launches / algorithmic passes (a loader row pass counts 32 or 16 B per point more)."""
    import csv, gzip, json, collections
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    rec = json.load(open(os.path.join(root, "profiles", "traffic.json")))["coupled8192"]
    rows = list(csv.reader(l for l in gzip.open(os.path.join(root, "profiles", "r02_fft_traffic.csv.gz"), "rt") if l.startswith('"')))
    hdr = rows[0]
    ik, im, iv, iid = hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Value"), hdr.index("ID")
    per = collections.OrderedDict()
    for r in rows[1:]:
        per.setdefault((r[iid], r[ik].split("(")[0].replace("void ", "")), {})[r[im]] = float(r[iv].replace(",", ""))
    total, npass = 0.0, 0.0
    for (_, name), d in per.items():
        total += d["dram__bytes_read.sum"] + d["dram__bytes_write.sum"]
        parts = name.rstrip(">").split(",")
        ld = int(parts[-1]) if name.startswith("k_fft_pass") and len(parts) == 6 else 0
        npass += {0: 1.0, 1: 2.0, 2: 1.5}[ld]
    assert len(per) == 2 * rec["transforms_captured"]
    assert abs(total / npass - rec["dram_bytes_per_pass"]) <= 1e-6 * rec["dram_bytes_per_pass"]
    assert 0.9 < rec["ratio"] <= 1.05
