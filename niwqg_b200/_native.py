"""ctypes binding of libniwqg_b200.so (C ABI declared in include/niwqg_b200.h).

There is no CPU fallback: if the shared library has not been built
(``python -c "import __graft_entry__ as g; g.build()"``) or no CUDA device is
present, model construction raises RuntimeError.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libniwqg_b200.so")
if os.environ.get("NIWQG_LIB"):          # development: an alternative build of the same library
    LIB_PATH = os.environ["NIWQG_LIB"]

MODEL_QG, MODEL_COUPLED, MODEL_UNCOUPLED, MODEL_YBJ, MODEL_QL = range(5)

# enum niwqg_field
FIELDS = ["Q", "QH", "PH", "P", "PHI", "PHIH", "PHIX", "PHIY", "LAPPHI", "U", "V", "QW", "QPSI", "QWH", "C", "CH",
          "FILTR", "EXPCH", "EXPCH_H", "QHCOEF", "F0", "FAB", "FC", "EXPCHW", "EXPCH_HW", "QHWCOEF", "F0W", "FABW",
          "FCW", "EXPCHC", "EXPCH_HC", "QHCCOEF", "F0C", "FABC", "FCC", "UV", "QS", "LAP2PHI", "UVQ"]
F = {n: i for i, n in enumerate(FIELDS)}
REAL_FIELDS = {"Q", "P", "U", "V", "QW", "QPSI", "C", "FILTR"}
PHYS_CPLX_FIELDS = {"PHI", "PHIX", "PHIY", "LAPPHI", "UV", "QS", "LAP2PHI", "UVQ"}
TABLE_FIELDS = set(FIELDS[F["FILTR"]:F["FCC"] + 1])
# the equation (q, phi, passive scalar c) each ETDRK4 table field belongs to, and the constructor keywords that set that
# equation's tables: the library gives an equation one table set per member when these differ between members
TABLE_EQ = dict([(n, "q") for n in FIELDS[F["EXPCH"]:F["FC"] + 1]] + [(n, "phi") for n in FIELDS[F["EXPCHW"]:F["FCW"] + 1]] +
                [(n, "c") for n in FIELDS[F["EXPCHC"]:F["FCC"] + 1]])
TABLE_KEYS = {"q": ("U", "nu4", "nu", "mu", "beta"), "phi": ("U", "f", "N", "m", "nu4w", "nuw", "muw"),
              "c": ("nu4c", "nuc", "muc")}

# enum niwqg_scalar
SCALARS = ["KE", "PW", "KW", "GAMMA1", "GAMMA2", "XI1", "XI2", "PI", "KE_QG", "ENS", "KE_NIW", "CKE_NIW", "IKE_NIW",
           "PE_NIW", "CONC", "SKEW", "EP_PHI", "EP_PSI", "CHI_Q", "CHI_PHI", "KE_QG_Q", "KE_QG_W", "KE_QG_QW", "CFL",
           "CVAR", "C2", "GRADC2", "GAMMA_C", "EP_C", "CHI_C"]
S = {n: i for i, n in enumerate(SCALARS)}
S_COUNT = len(SCALARS)

FFT_C2C_FWD, FFT_C2C_INV, FFT_R2C, FFT_C2R, FFT_R2C_FULL = range(5)
JAC_PSI_Q, JAC_PHIC_PHI, JAC_PSI_PHI = range(3)

EXPORTS = ["niwqg_create", "niwqg_destroy", "niwqg_last_error", "niwqg_set_q", "niwqg_set_phi", "niwqg_set_c",
           "niwqg_step", "niwqg_diagnostics", "niwqg_status", "niwqg_get_scalars", "niwqg_get_field",
           "niwqg_field_bytes", "niwqg_fft2", "niwqg_jacobian", "niwqg_sync", "niwqg_time_steps",
           "niwqg_launch_count", "niwqg_stream", "niwqg_profile", "niwqg_nccl_unique_id", "niwqg_ic",
           "niwqg_get_field_async", "niwqg_wait_transfers", "niwqg_stage_q", "niwqg_stage_phi",
           "niwqg_ipc_export", "niwqg_ipc_import", "niwqg_ipc_disable", "niwqg_state_slots", "niwqg_set_field",
           "niwqg_carry_count", "niwqg_get_carry", "niwqg_set_carry", "niwqg_create_ensemble",
           "niwqg_particles_set", "niwqg_particles_count", "niwqg_particles_get", "niwqg_particles_sample"]


class Params(C.Structure):
    _fields_ = [("struct_size", C.c_size_t),
                ("model", C.c_int), ("nx", C.c_int), ("batch", C.c_int), ("device", C.c_int),
                ("L", C.c_double), ("dt", C.c_double), ("U", C.c_double), ("f", C.c_double), ("N", C.c_double),
                ("m", C.c_double), ("nu", C.c_double), ("nu4", C.c_double), ("mu", C.c_double),
                ("nuw", C.c_double), ("nu4w", C.c_double), ("muw", C.c_double), ("beta", C.c_double),
                ("use_filter", C.c_int), ("dealias", C.c_int), ("passive_scalar", C.c_int),
                ("nu4c", C.c_double), ("nuc", C.c_double), ("muc", C.c_double),
                ("rank", C.c_int), ("nranks", C.c_int), ("nccl_id", C.c_ubyte * 128)]


# the coefficients one ensemble member may set for itself (struct niwqg_member_params)
MEMBER_KEYS = ("U", "f", "N", "m", "nu", "nu4", "mu", "nuw", "nu4w", "muw", "beta", "nu4c", "nuc", "muc")


class MemberParams(C.Structure):
    _fields_ = [("struct_size", C.c_size_t)] + [(k, C.c_double) for k in MEMBER_KEYS]


def member_keywords(batch, per_member, shared):
    """Validate the constructor keywords of a model with ``batch`` members.  ``per_member``: {name: value}, each a
    scalar (all members share it; returned unchanged) or a sequence of ``batch`` values (returned as a float64 array).
    ``shared``: {name: value} that every member has in common, so a sequence there is an error.  ValueError names the
    keyword."""
    for k, v in shared.items():
        if np.ndim(v) != 0:
            raise ValueError("%s is common to all members of an ensemble: give one value, not a sequence" % k)
    out = {}
    for k, v in per_member.items():
        if np.ndim(v) == 0:
            out[k] = v
            continue
        a = np.asarray(v, dtype=np.float64)
        if a.ndim != 1 or a.size != batch:
            raise ValueError("%s: expected one value or a sequence of batch=%d values, got shape %s"
                             % (k, batch, np.shape(v)))
        out[k] = a
    return out


_lib = None


def load():
    """Load the shared library (once).  Raises RuntimeError when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("niwqg_b200: %s not built (run __graft_entry__.build()); there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, ip, dp = C.c_void_p, C.c_int, C.POINTER(C.c_double)
    lib.niwqg_create.argtypes = [C.POINTER(Params), C.POINTER(vp)]
    lib.niwqg_create_ensemble.argtypes = [C.POINTER(Params), C.POINTER(MemberParams), C.POINTER(vp)]
    lib.niwqg_destroy.argtypes = [vp]
    lib.niwqg_last_error.argtypes = [vp]
    lib.niwqg_last_error.restype = C.c_char_p
    for n in ("niwqg_set_q", "niwqg_set_phi", "niwqg_set_c"):
        getattr(lib, n).argtypes = [vp, vp, ip]
    for n in ("niwqg_stage_q", "niwqg_stage_phi"):
        getattr(lib, n).argtypes = [vp, vp]
    lib.niwqg_ic.argtypes = [vp, ip, vp, ip, vp]
    lib.niwqg_step.argtypes = [vp, ip]
    for n in ("niwqg_diagnostics", "niwqg_status", "niwqg_get_scalars"):
        getattr(lib, n).argtypes = [vp, vp]
    lib.niwqg_get_field.argtypes = [vp, ip, ip, vp, C.c_size_t, ip]
    lib.niwqg_get_field_async.argtypes = [vp, ip, ip, vp, C.c_size_t]
    lib.niwqg_wait_transfers.argtypes = [vp]
    lib.niwqg_field_bytes.argtypes = [vp, ip]
    lib.niwqg_field_bytes.restype = C.c_size_t
    lib.niwqg_fft2.argtypes = [vp, vp, vp, ip]
    lib.niwqg_jacobian.argtypes = [vp, ip, vp]
    lib.niwqg_sync.argtypes = [vp]
    lib.niwqg_time_steps.argtypes = [vp, ip, C.POINTER(C.c_float)]
    lib.niwqg_launch_count.argtypes = [vp]
    lib.niwqg_launch_count.restype = C.c_longlong
    lib.niwqg_profile.argtypes = [vp, ip, vp, vp]
    lib.niwqg_stream.argtypes = [vp]
    lib.niwqg_stream.restype = vp
    lib.niwqg_nccl_unique_id.argtypes = [vp]
    lib.niwqg_ipc_export.argtypes = [vp, vp, C.c_size_t]
    lib.niwqg_ipc_import.argtypes = [vp, vp, C.c_size_t]
    lib.niwqg_ipc_disable.argtypes = [vp]
    lib.niwqg_state_slots.argtypes = [vp, vp, ip]
    lib.niwqg_set_field.argtypes = [vp, ip, ip, vp, C.c_size_t, ip]
    lib.niwqg_carry_count.argtypes = [vp]
    lib.niwqg_get_carry.argtypes = [vp, vp]
    lib.niwqg_set_carry.argtypes = [vp, vp]
    lib.niwqg_particles_set.argtypes = [vp, vp, ip, C.c_double, ip, ip]
    lib.niwqg_particles_count.argtypes = [vp]
    lib.niwqg_particles_get.argtypes = [vp, vp, vp]
    lib.niwqg_particles_sample.argtypes = [vp, ip, vp]
    _lib = lib
    return lib


def _nccl_library_path():
    """The NCCL that ships with torch (site-packages/nvidia/nccl/lib); None = leave it to the dynamic loader."""
    if os.environ.get("NIWQG_NCCL_LIB"):
        return os.environ["NIWQG_NCCL_LIB"]
    try:
        import nvidia.nccl as _n
        for d in list(_n.__path__):
            cand = os.path.join(d, "lib", "libnccl.so.2")
            if os.path.exists(cand):
                return cand
    except Exception:
        pass
    return None


def nccl_unique_id():
    """128-byte ncclUniqueId (call on rank 0, broadcast to the other ranks, pass as nccl_id=...)."""
    path = _nccl_library_path()
    if path:
        os.environ["NIWQG_NCCL_LIB"] = path
    lib = load()
    buf = C.create_string_buffer(128)
    rc = lib.niwqg_nccl_unique_id(buf)
    if rc != 0:
        msg = lib.niwqg_last_error(None)
        raise RuntimeError("niwqg_nccl_unique_id failed (%d): %s" % (rc, msg.decode() if msg else "?"))
    return buf.raw


# ---- slab column map (mirror of struct Grid in csrc/common.cuh); pure Python so that CPU tests can check it
def slab_kx(N, nranks, rank):
    """Global column index kx of every local spectral column of `rank` (length N/nranks)."""
    if nranks == 1:
        return np.arange(N)
    h = N // (2 * nranks)
    lc = np.arange(2 * h)
    kx = np.where(lc < h, rank * h + lc, N - (rank * h + lc - h))
    if rank == 0:
        kx[h] = N // 2
    return kx


def slab_owner(N, nranks, kx):
    """(rank, local column) that holds global column kx."""
    h = N // (2 * nranks)
    if kx < N // 2:
        return kx // h, kx % h
    if kx == N // 2:
        return 0, h
    m = N - kx
    return m // h, h + m % h


# fields niwqg_particles_sample interpolates, by the name Model.sample_particles takes
PARTICLE_FIELDS = {"q": "Q", "u": "U", "v": "V", "phi": "PHI"}


def particle_positions(xy, batch):
    """Validate the positions given to set_particles: (P, 2) seeds every member, (batch, P, 2) each member its own.
    Returns a C-contiguous float64 (batch, P, 2) array.  ValueError for another shape or a non-finite value."""
    a = np.asarray(xy)
    if a.dtype.kind not in "iuf":
        raise ValueError("particle positions must be real numbers, got dtype %s" % a.dtype)
    a = a.astype(np.float64)
    if a.ndim == 2 and a.shape[1] == 2:
        a = np.broadcast_to(a[None], (batch,) + a.shape)
    if a.ndim != 3 or a.shape[0] != batch or a.shape[2] != 2 or a.shape[1] == 0:
        raise ValueError("particle positions must have shape (P, 2) or (batch=%d, P, 2) with P >= 1, got %s"
                         % (batch, np.shape(xy)))
    if a.shape[1] > 2 ** 31 - 1:
        raise ValueError("at most 2**31 - 1 particles per member")
    if not np.all(np.isfinite(a)):
        raise ValueError("particle positions must be finite")
    return np.ascontiguousarray(a)


class Handle(object):
    """Owns one niwqg_handle.  Every method raises RuntimeError on a non-zero return.  A keyword of MEMBER_KEYS given
    as an array of ``batch`` values gives every member its own value (niwqg_create_ensemble)."""

    def __init__(self, **kw):
        path = _nccl_library_path() if kw.get("nranks", 1) > 1 else None
        if path:
            os.environ["NIWQG_NCCL_LIB"] = path
        self.lib = load()
        p = Params()
        p.struct_size = C.sizeof(Params)
        swept = {k: np.asarray(v, np.float64) for k, v in kw.items() if k in MEMBER_KEYS and np.ndim(v) != 0}
        for k, v in kw.items():
            if k == "nccl_id":      # raw 128 bytes (a c_char array would stop at the first NUL)
                if v is None or len(v) != 128:
                    raise ValueError("nccl_id must be the 128 bytes of nccl_unique_id()")
                C.memmove(C.addressof(p) + Params.nccl_id.offset, bytes(v), 128)
            else:
                setattr(p, k, float(swept[k][0]) if k in swept else v)
        members = None
        if swept:
            for k, v in swept.items():
                if v.shape != (p.batch,):
                    raise ValueError("%s: expected %d per-member values, got shape %s" % (k, p.batch, v.shape))
            members = (MemberParams * p.batch)()
            for b in range(p.batch):
                members[b].struct_size = C.sizeof(MemberParams)
                for k in MEMBER_KEYS:
                    setattr(members[b], k, float(swept[k][b]) if k in swept else getattr(p, k))
        # equations whose tables the library holds per member (its rule: the equation's keywords differ)
        eqs = ("q", "c") if p.model == MODEL_QG else ("q", "phi")
        self.table_members = {eq for eq in eqs if any(k in swept and np.any(swept[k] != swept[k][0]) for k in TABLE_KEYS[eq])}
        self.params = p
        self._staged = {}
        self.h = C.c_void_p()
        rc = self.lib.niwqg_create_ensemble(C.byref(p), members, C.byref(self.h))
        if rc != 0:
            msg = self.lib.niwqg_last_error(None)
            self.h = None
            raise RuntimeError("niwqg_create failed (%d): %s" % (rc, msg.decode() if msg else "?"))
        self.N, self.B = p.nx, p.batch
        self.nranks, self.rank = max(1, p.nranks), (p.rank if p.nranks > 1 else 0)
        self.nyl = p.nx // self.nranks            # local physical rows
        self.nk = p.nx // 2 + 1 if p.model == MODEL_QG else p.nx // self.nranks   # local spectral columns

    def _ck(self, rc):
        if rc != 0:
            msg = self.lib.niwqg_last_error(self.h)
            raise RuntimeError("niwqg_b200 error %d: %s" % (rc, msg.decode() if msg else "?"))

    def close(self):
        if getattr(self, "h", None):
            self.lib.niwqg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- slab: fused exchange over peer memory ------------------------------
    IPC_BYTES = 256      # 2 lanes x 2 receive buffers x 64-byte cudaIpcMemHandle_t

    def ipc_export(self):
        buf = C.create_string_buffer(self.IPC_BYTES)
        self._ck(self.lib.niwqg_ipc_export(self.h, buf, self.IPC_BYTES))
        return buf.raw

    def ipc_import(self, all_ranks_bytes):
        if len(all_ranks_bytes) != self.IPC_BYTES * self.nranks:
            raise ValueError("expected %d bytes of IPC handles" % (self.IPC_BYTES * self.nranks))
        self._ck(self.lib.niwqg_ipc_import(self.h, all_ranks_bytes, self.IPC_BYTES))

    def ipc_disable(self):
        self._ck(self.lib.niwqg_ipc_disable(self.h))

    # -- seeding -----------------------------------------------------------
    def _host(self, a, dtype):
        a = np.ascontiguousarray(a, dtype=dtype)
        if self.nranks > 1 and a.size == self.N * self.N:      # whole-grid array: keep this rank's rows
            a = np.ascontiguousarray(a.reshape(self.N, self.N)[self.rank * self.nyl:(self.rank + 1) * self.nyl])
        want = self.B * self.nyl * self.N
        if a.size != want:
            if a.size == self.N * self.N and self.B > 1:
                a = np.ascontiguousarray(np.broadcast_to(a.reshape(1, self.N, self.N), (self.B, self.N, self.N)))
            else:
                raise ValueError("expected %d values, got %d" % (want, a.size))
        return a

    # The library returns from set_* once the host array has been copied (the caller may reuse it); the inversion and
    # transforms that follow stay queued on the handle's stream, and every later call is ordered behind them.
    # q / phi None: seed from the array queued by stage_q / stage_phi (uploaded while the device was busy).
    def set_q(self, q=None):
        if q is None:
            self._ck(self.lib.niwqg_set_q(self.h, None, 0))
            self._staged.pop("q", None)
            return
        a = self._host(q, np.float64)
        self._ck(self.lib.niwqg_set_q(self.h, a.ctypes.data, 0))

    def set_phi(self, phi=None):
        if phi is None:
            self._ck(self.lib.niwqg_set_phi(self.h, None, 0))
            self._staged.pop("phi", None)
            return
        a = self._host(phi, np.complex128)
        self._ck(self.lib.niwqg_set_phi(self.h, a.ctypes.data, 0))

    def stage_q(self, q):
        """Queue the upload of the next set_q() input (niwqg_stage_q): returns at once; the array is kept alive here
        and must not be written to until set_q() has returned."""
        a = self._host(q, np.float64)
        self._staged["q"] = a
        self._ck(self.lib.niwqg_stage_q(self.h, a.ctypes.data))

    def stage_phi(self, phi):
        a = self._host(phi, np.complex128)
        self._staged["phi"] = a
        self._ck(self.lib.niwqg_stage_phi(self.h, a.ctypes.data))

    def set_c(self, c):
        a = self._host(c, np.float64)
        self._ck(self.lib.niwqg_set_c(self.h, a.ctypes.data, 0))

    IC_KINDS = {"LambDipole": 0, "McWilliams1984": 1, "Danioux2015": 2, "WavePacket": 3, "PlaneWave": 4, "Uniform": 5}

    def ic(self, kind, params, rand01=None):
        """Generate an initial condition on the device and seed the model with it (niwqg_ic)."""
        prm = np.ascontiguousarray(params, dtype=np.float64)
        r = None
        if rand01 is not None:
            r = np.ascontiguousarray(rand01, dtype=np.float64)
            if r.size != self.N * self.N:
                raise ValueError("rand01 must hold N*N uniform numbers")
        self._ck(self.lib.niwqg_ic(self.h, self.IC_KINDS[kind], prm.ctypes.data, prm.size, r.ctypes.data if r is not None else None))
        self.sync()

    def set_q_device(self, ptr):
        self._ck(self.lib.niwqg_set_q(self.h, C.c_void_p(ptr), 1))

    def set_phi_device(self, ptr):
        self._ck(self.lib.niwqg_set_phi(self.h, C.c_void_p(ptr), 1))

    # -- stepping ----------------------------------------------------------
    def step(self, n=1):
        self._ck(self.lib.niwqg_step(self.h, int(n)))

    def time_steps(self, n):
        ms = C.c_float()
        self._ck(self.lib.niwqg_time_steps(self.h, int(n), C.byref(ms)))
        return ms.value

    def sync(self):
        self._ck(self.lib.niwqg_sync(self.h))

    PROFILE_KINDS = ("fft_row", "fft_col", "phys", "spec", "small", "comm", "fft_p", "fft_row_ld", "fft_row_ld2")

    def profile(self, enable):
        """Switch per-kernel-kind event timing on/off; returns {kind: (total_ms, launches)} recorded so far."""
        ms = np.zeros(len(self.PROFILE_KINDS))
        cnt = np.zeros(len(self.PROFILE_KINDS), np.int64)
        self._ck(self.lib.niwqg_profile(self.h, int(bool(enable)), ms.ctypes.data, cnt.ctypes.data))
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(self.PROFILE_KINDS)}

    def field_into(self, name, out, member=0, wait=True):
        """Copy one member's field into a caller-provided (e.g. pinned) host array.  wait=False queues the copy on the
        handle's copy stream and returns at once; the array is valid after wait_transfers() (or sync())."""
        if wait:
            self._ck(self.lib.niwqg_get_field(self.h, F[name], member, out.ctypes.data, out.nbytes, 0))
        else:
            self._ck(self.lib.niwqg_get_field_async(self.h, F[name], member, out.ctypes.data, out.nbytes))
        return out

    def wait_transfers(self):
        self._ck(self.lib.niwqg_wait_transfers(self.h))

    def launch_count(self):
        return int(self.lib.niwqg_launch_count(self.h))

    # -- reads -------------------------------------------------------------
    def scalars(self, which="scalars"):
        out = np.zeros((self.B, S_COUNT))
        fn = {"scalars": self.lib.niwqg_get_scalars, "diagnostics": self.lib.niwqg_diagnostics}[which]
        self._ck(fn(self.h, out.ctypes.data))
        return out

    def status(self):
        out = np.zeros((self.B, 4))
        self._ck(self.lib.niwqg_status(self.h, out.ctypes.data))
        return out

    def field(self, name, member=None):
        fid = F[name]
        N, nk = self.N, self.nk
        if name in REAL_FIELDS:
            shape, dt = ((N, nk) if name == "FILTR" else (self.nyl, N)), np.float64
        elif name in PHYS_CPLX_FIELDS:
            shape, dt = (self.nyl, N), np.complex128
        else:
            shape, dt = (N, nk), np.complex128
        if name in TABLE_FIELDS:     # shared tables: one array; per-member tables: a member axis as for the state
            pm = TABLE_EQ.get(name) in self.table_members
            members = (range(self.B) if member is None else [member]) if pm else [0]
        else:
            members = range(self.B) if member is None else [member]
        outs = []
        for mm in members:
            a = np.empty(shape, dt)
            self._ck(self.lib.niwqg_get_field(self.h, fid, mm, a.ctypes.data, a.nbytes, 0))
            outs.append(a)
        if len(outs) == 1:
            return outs[0]
        return np.stack(outs)

    # -- checkpoint / exact restart ---------------------------------------
    def state_slots(self):
        """Names of the fields that make up this handle's state (niwqg_state_slots)."""
        ids = np.zeros(16, np.int32)
        n = self.lib.niwqg_state_slots(self.h, ids.ctypes.data, ids.size)
        if n < 0:
            raise RuntimeError("niwqg_state_slots: more than %d slots" % ids.size)
        return [FIELDS[i] for i in ids[:n]]

    def set_field(self, name, member, a):
        """Write one member's state slot, in the layout field() returns it (niwqg_set_field)."""
        a = np.ascontiguousarray(a, np.float64 if name in REAL_FIELDS else np.complex128)
        self._ck(self.lib.niwqg_set_field(self.h, F[name], member, a.ctypes.data, a.nbytes, 0))

    def carry(self):
        out = np.zeros(self.lib.niwqg_carry_count(self.h))
        self._ck(self.lib.niwqg_get_carry(self.h, out.ctypes.data))
        return out

    def set_carry(self, a):
        a = np.ascontiguousarray(a, np.float64)
        if a.size != self.lib.niwqg_carry_count(self.h):
            raise ValueError("expected %d carry values, got %d" % (self.lib.niwqg_carry_count(self.h), a.size))
        self._ck(self.lib.niwqg_set_carry(self.h, a.ctypes.data))

    # -- Lagrangian particles ---------------------------------------------
    def particles_set(self, xy, t, waves):
        """xy: (batch, P, 2) float64 as particle_positions returns it, or None to remove the particles."""
        if xy is None:
            self._ck(self.lib.niwqg_particles_set(self.h, None, 0, float(t), 0, 0))
            return
        self._ck(self.lib.niwqg_particles_set(self.h, xy.ctypes.data, xy.shape[1], float(t), int(bool(waves)), 0))

    def particles_count(self):
        return int(self.lib.niwqg_particles_count(self.h))

    def particles(self):
        """(positions (batch, P, 2), clock), or (None, None) without particles."""
        n = self.particles_count()
        if n == 0:
            return None, None
        xy = np.empty((self.B, n, 2))
        t = np.zeros(1)
        self._ck(self.lib.niwqg_particles_get(self.h, xy.ctypes.data, t.ctypes.data))
        return xy, float(t[0])

    def particles_sample(self, name):
        n = self.particles_count()
        out = np.empty((self.B, n), np.complex128 if name == "PHI" else np.float64)
        self._ck(self.lib.niwqg_particles_sample(self.h, F[name], out.ctypes.data))
        return out

    def field_to_device(self, name, member, ptr, nbytes):
        self._ck(self.lib.niwqg_get_field(self.h, F[name], member, C.c_void_p(ptr), nbytes, 1))

    def fft2(self, x, kind):
        N, nh = self.N, self.N // 2 + 1
        if kind in (FFT_R2C, FFT_R2C_FULL):
            a = np.ascontiguousarray(x, np.float64)
            out = np.empty((N, nh) if kind == FFT_R2C else (N, N), np.complex128)
        elif kind == FFT_C2R:
            a = np.ascontiguousarray(x, np.complex128)
            if a.shape != (N, nh):
                raise ValueError("irfft2 input must be (%d,%d)" % (N, nh))
            out = np.empty((N, N), np.float64)
        else:
            a = np.ascontiguousarray(x, np.complex128)
            out = np.empty((N, N), np.complex128)
        if self.nranks > 1:
            # slab: forward takes this rank's rows (nyl, N) and returns its column slab (N, ncl); inverse the reverse
            fwd = kind in (FFT_C2C_FWD, FFT_R2C_FULL)
            want = (self.nyl, N) if fwd else (N, self.nk)
            if a.shape != want:
                raise ValueError("slab fft input must be %s" % (want,))
            out = np.empty((N, self.nk) if fwd else (self.nyl, N), np.complex128)
        elif kind != FFT_C2R and a.shape != (N, N):
            raise ValueError("fft input must be (%d,%d)" % (N, N))
        self._ck(self.lib.niwqg_fft2(self.h, a.ctypes.data, out.ctypes.data, kind))
        return out

    def jacobian(self, which):
        out = np.empty((self.N, self.nk), np.complex128)
        self._ck(self.lib.niwqg_jacobian(self.h, which, out.ctypes.data))
        return out
