"""Checkpoint and exact restart (DESIGN.md section 6b).

A checkpoint is a directory::

    checkpoint.json    format, version, model class, constructor keywords, nx, batch, t, tc, host status attributes,
                       the state slots (name, dtype, shape) and the scalar carry
    <SLOT>.npy         one per state slot, whole grid in natural order with a leading member axis:
                       (batch, nx, nx), or (batch, nx, nx/2+1) for the QG half spectrum
    diagnostics.npz    the 'value' array of every diagnostic that has one
    PARTICLES.npy      only for a model with Lagrangian particles: their unwrapped positions, (batch, P, 2); the
                       ``particles`` entry of checkpoint.json holds P, the particle clock and ``waves``

Which buffers make up the state is decided by the CUDA library (niwqg_state_slots); this module only moves them
between the device and the files.  Fields are streamed one member at a time, so the host never holds more than one
field.  A slab run writes and reads in parallel: every rank moves its own rows (physical fields) or its own columns
(spectral fields, ``slab_kx``) of the same memory-mapped files, which is what makes a checkpoint portable between one
GPU and any number of ranks.

The device side is reached through an object with the interface of :class:`HandleIO` (``nx``, ``batch``, ``rank``,
``nranks``, ``slots``, ``read``, ``write``, ``get_carry``, ``set_carry``, ``agree``), so the file layer runs without a
GPU as well.
"""
import json
import os
import shutil
import warnings

import numpy as np

from . import _native as nat

FORMAT = "niwqg_b200-checkpoint"
VERSION = 1
META = "checkpoint.json"
DIAGNOSTICS = "diagnostics.npz"
PARTICLES = "PARTICLES"
STATUS_ATTRS = ("ke", "kew", "pew", "cfl")


class Slot(object):
    """One state slot: ``shape`` is the whole-grid shape of one member; ``split`` says how a slab run divides it
    ('rows': physical rows, 'cols': spectral columns in the conjugate-symmetric ownership of ``slab_kx``)."""

    def __init__(self, name, dtype, shape, split):
        self.name, self.dtype, self.shape, self.split = name, np.dtype(dtype), tuple(shape), split


class HandleIO(object):
    """Device side of a checkpoint for a model's native handle.  ``dist`` (torch.distributed) connects the ranks of a
    slab run."""

    def __init__(self, model, dist=None):
        self.h = model._h
        self.nx, self.batch = model.nx, model.batch
        self.rank, self.nranks = self.h.rank, self.h.nranks
        self.dist = dist

    def slots(self):
        out = []
        for name in self.h.state_slots():
            if name in nat.REAL_FIELDS or name in nat.PHYS_CPLX_FIELDS:
                dt = np.float64 if name in nat.REAL_FIELDS else np.complex128
                out.append(Slot(name, dt, (self.nx, self.nx), "rows"))
            else:
                nk = self.nx // 2 + 1 if self.h.params.model == nat.MODEL_QG else self.nx
                out.append(Slot(name, np.complex128, (self.nx, nk), "cols"))
        return out

    def read(self, name, member):
        return self.h.field(name, member)

    def write(self, name, member, a):
        self.h.set_field(name, member, a)

    def get_carry(self):
        return self.h.carry()

    def set_carry(self, a):
        self.h.set_carry(a)

    def agree(self, ok):
        """Barrier that also tells every rank whether all of them got there without an error."""
        return agree(self.dist, self.nranks, ok)


def agree(dist, nranks, ok):
    """True on every rank when ``ok`` is true on every rank (one all-reduce over ``dist``); ``ok`` itself on one rank."""
    if nranks == 1:
        return bool(ok)
    import torch
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    t = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(t.item())


def _local_index(slot, io):
    """Index of this rank's part within one member's whole-grid array."""
    if io.nranks == 1:
        return slice(None)
    if slot.split == "rows":
        n = slot.shape[0] // io.nranks
        return slice(io.rank * n, (io.rank + 1) * n)
    return (slice(None), nat.slab_kx(slot.shape[0], io.nranks, io.rank))


def _file(path, name):
    return os.path.join(path, name + ".npy")


def _aside(path, what):
    return os.path.join(os.path.dirname(path), "." + os.path.basename(path) + what)


def _step(io, fn):
    """Run ``fn`` (on this rank), then wait for every rank; raise on all of them if it failed on any."""
    err = None
    try:
        fn()
    except Exception as e:          # re-raised below, after the other ranks have been told
        err = e
    if not io.agree(err is None):
        raise err if err is not None else RuntimeError("writing the checkpoint failed on another rank")


def write(path, meta, io, diagnostics=None, arrays=None):
    """Write the state behind ``io`` and the host-side ``meta`` (a JSON-able dict) as the checkpoint ``path``.

    ``path`` must not exist, be an empty directory or hold a checkpoint: any other directory is refused before anything
    is written, so a data directory is never replaced.  Everything goes to the temporary sibling ``.<name>.partial``
    first, which replaces ``path`` only once it is complete: a failure while saving leaves the previous checkpoint as
    it was.  Replacing a directory takes two renames (``path`` -> ``.<name>.old``, ``.<name>.partial`` -> ``path``);
    if the process dies between them, ``locate`` finds the previous checkpoint under ``.<name>.old``.  In a slab run
    every rank calls this; rank 0 creates the files and does the replacing, and an error on any rank is raised on all
    of them.  ``arrays``: {name: array} written by rank 0 as ``<name>.npy`` beside the slots."""
    path = os.path.abspath(path)
    tmp, old = _aside(path, ".partial"), _aside(path, ".old")
    slots = io.slots()

    def refuse_foreign():
        if os.path.exists(path) and not (os.path.isdir(path) and
                                         (not os.listdir(path) or os.path.exists(os.path.join(path, META)))):
            raise ValueError("%s exists and is not a checkpoint: refusing to replace it" % path)

    def create():
        if os.path.exists(tmp):
            shutil.rmtree(tmp)
        os.makedirs(tmp)
        for s in slots:
            np.lib.format.open_memmap(_file(tmp, s.name), mode="w+", dtype=s.dtype, shape=(io.batch,) + s.shape).flush()

    def fill():
        for s in slots:
            idx = _local_index(s, io)
            for m in range(io.batch):
                mm = np.load(_file(tmp, s.name), mmap_mode="r+")
                mm[m][idx] = io.read(s.name, m)
                mm.flush()
                del mm

    def finish():
        full = dict(meta, format=FORMAT, version=VERSION, nx=io.nx, batch=io.batch,
                    slots=[dict(name=s.name, dtype=s.dtype.str, shape=[io.batch] + list(s.shape)) for s in slots],
                    carry=[float(v) for v in io.get_carry()])
        if diagnostics:
            np.savez(os.path.join(tmp, DIAGNOSTICS), **diagnostics)
        for name, a in (arrays or {}).items():
            np.save(_file(tmp, name), a)
        with open(os.path.join(tmp, META), "w") as f:
            json.dump(full, f, indent=1)
            f.flush()
            os.fsync(f.fileno())
        if os.path.exists(path):
            # a directory cannot replace a non-empty one in one rename: move the old one aside, then drop it
            if os.path.exists(old):
                shutil.rmtree(old)
            os.replace(path, old)
        os.replace(tmp, path)
        if os.path.exists(old):
            shutil.rmtree(old)

    _step(io, refuse_foreign)       # every rank sees the same directory: all refuse together
    _step(io, create if io.rank == 0 else (lambda: None))
    _step(io, fill)
    _step(io, finish if io.rank == 0 else (lambda: None))


def locate(path):
    """The directory that holds the checkpoint ``path``: ``path`` itself, or ``.<name>.old`` beside it when a save died
    between the two renames of its replacement."""
    path = os.path.abspath(path)
    if not os.path.exists(os.path.join(path, META)) and os.path.exists(os.path.join(_aside(path, ".old"), META)):
        warnings.warn("%s: using the previous checkpoint %s left by an interrupted save" % (path, _aside(path, ".old")))
        return _aside(path, ".old")
    return path


def read_meta(path):
    """The checkpoint's ``checkpoint.json``, after checking its format and version."""
    fn = os.path.join(path, META)
    if not os.path.exists(fn):
        raise FileNotFoundError("%s is not a checkpoint (no %s)" % (path, META))
    with open(fn) as f:
        meta = json.load(f)
    if meta.get("format") != FORMAT:
        raise ValueError("%s: not a %s" % (fn, FORMAT))
    if meta.get("version") != VERSION:
        raise ValueError("%s: checkpoint format version %r, this library reads version %d"
                         % (fn, meta.get("version"), VERSION))
    return meta


def check(path, meta, io):
    """Raise unless every slot ``io`` needs is in the checkpoint with the right dtype and shape.  Reads no data."""
    if meta["nx"] != io.nx or meta["batch"] != io.batch:
        raise ValueError("checkpoint has nx=%d, batch=%d; the model has nx=%d, batch=%d"
                         % (meta["nx"], meta["batch"], io.nx, io.batch))
    saved = {s["name"] for s in meta["slots"]}
    for s in io.slots():
        if s.name not in saved:
            raise ValueError("checkpoint %s has no state slot %s, which this model carries (for YBJ / QL: LAP2PHI exists "
                             "only with nu4w != 0, so nu4w cannot be switched on at a restart)" % (path, s.name))
        fn = _file(path, s.name)
        if not os.path.exists(fn):
            raise FileNotFoundError("checkpoint %s: missing %s" % (path, os.path.basename(fn)))
        mm = np.load(fn, mmap_mode="r")
        if mm.dtype != s.dtype or mm.shape != (io.batch,) + s.shape:
            raise ValueError("checkpoint %s: %s is %s %s, expected %s %s"
                             % (path, os.path.basename(fn), mm.dtype, mm.shape, s.dtype, (io.batch,) + s.shape))
        del mm
    if len(meta["carry"]) != len(io.get_carry()):
        raise ValueError("checkpoint %s: %d carry values, the model has %d" % (path, len(meta["carry"]), len(io.get_carry())))


def read(path, meta, io):
    """Stream the checkpoint's state into the device behind ``io`` (call ``check`` first).  Returns the diagnostics
    arrays."""
    for s in io.slots():
        idx = _local_index(s, io)
        for m in range(io.batch):
            mm = np.load(_file(path, s.name), mmap_mode="r")
            io.write(s.name, m, mm[m][idx])
            del mm
    io.set_carry(np.array(meta["carry"], np.float64))
    fn = os.path.join(path, DIAGNOSTICS)
    if not os.path.exists(fn):
        return {}
    with np.load(fn) as z:
        return {k: z[k] for k in z.files}


# ---------------------------------------------------------------------------- model level
def _class_name(cls):
    return cls.__module__ + "." + cls.__qualname__


def _keywords(model, names):
    """The model's keywords as JSON values: a per-member keyword (an array) becomes a list."""
    out = {}
    for k in names:
        v = getattr(model, model._checkpoint_attr.get(k, k))
        out[k] = v.tolist() if isinstance(v, np.ndarray) else (v.item() if isinstance(v, np.generic) else v)
    return out


def _same(a, b):
    """Keyword values a == b; lists (per-member values) element by element, and never equal to a scalar."""
    if isinstance(a, (list, np.ndarray)) or isinstance(b, (list, np.ndarray)):
        return np.shape(a) == np.shape(b) and bool(np.all(np.asarray(a) == np.asarray(b)))
    return a == b


def _io(model, dist):
    if model._h.nranks > 1 and dist is None:
        import torch.distributed as dist
    return HandleIO(model, dist)


def save(model, path, dist=None):
    """Write ``model``'s state as the checkpoint ``path`` (``Model.save_checkpoint``)."""
    status = {}
    for k in STATUS_ATTRS:
        v = model._ke if k == "ke" and hasattr(type(model), "_ke") else model.__dict__.get(k)
        if v is not None:
            status[k] = np.asarray(v).tolist()
    meta = dict(model=_class_name(type(model)), params=_keywords(model, model._checkpoint_params),
                run=_keywords(model, model._checkpoint_run), t=model.t, tc=model.tc, status=status)
    diags = {k: d["value"] for k, d in model.diagnostics.items() if "value" in d}
    arrays = {}
    ps = model._particles_state()
    if ps is not None:
        xy, t, waves = ps
        meta["particles"] = dict(count=int(xy.shape[1]), t=t, waves=bool(waves))
        arrays[PARTICLES] = xy
    write(path, meta, _io(model, dist), diags, arrays)


def load(model, path, dist=None, changed=()):
    """Restore the checkpoint ``path`` into ``model`` (``Model.load_checkpoint``).  The model must be of the same class,
    grid and ensemble size, with the same arithmetic parameters except those named in ``changed``; every check runs
    before anything on the model changes."""
    path = locate(path)
    meta = read_meta(path)
    diffs = []
    if meta["model"] != _class_name(type(model)):
        diffs.append("class %s (model: %s)" % (meta["model"], _class_name(type(model))))
    for k in ("nx", "batch"):
        if meta[k] != getattr(model, k):
            diffs.append("%s=%r (model: %r)" % (k, meta[k], getattr(model, k)))
    mine = _keywords(model, model._checkpoint_params)
    for k, v in sorted(meta["params"].items()):
        if k not in changed and not _same(mine.get(k), v):
            diffs.append("%s=%r (model: %r)" % (k, v, mine.get(k)))
    if diffs:
        raise ValueError("checkpoint %s does not match the model: %s" % (path, ", ".join(diffs)))
    io = _io(model, dist)
    check(path, meta, io)
    xy = _check_particles(path, meta, model)
    values = read(path, meta, io)
    model.t, model.tc = meta["t"], meta["tc"]
    for name, d in model.diagnostics.items():
        if name in values:
            d["value"] = values[name]
        else:
            d.pop("value", None)
    if xy is not None:
        pm = meta["particles"]
        model._set_particles_state(xy, pm["t"], pm["waves"])
    elif model._particles_state() is not None:
        model.set_particles(None)       # the saved run had none
    for k in STATUS_ATTRS:
        v = meta["status"].get(k)
        v = None if v is None else (np.array(v) if isinstance(v, list) else v)
        if k == "ke" and hasattr(type(model), "_ke"):
            model._ke = v
        elif v is None:
            model.__dict__.pop(k, None)
        else:
            setattr(model, k, v)


def _check_particles(path, meta, model):
    """The saved particle positions (batch, P, 2), or None when the checkpoint has no particles.  Reads and checks them
    before anything on the model changes."""
    pm = meta.get("particles")
    if pm is None:
        return None
    if model._h.nranks > 1:
        raise NotImplementedError("checkpoint %s has Lagrangian particles: a slab-decomposed model cannot carry them"
                                  % path)
    fn = _file(path, PARTICLES)
    if not os.path.exists(fn):
        raise FileNotFoundError("checkpoint %s: missing %s" % (path, os.path.basename(fn)))
    xy = np.load(fn)
    if xy.dtype != np.float64 or xy.shape != (model.batch, pm["count"], 2):
        raise ValueError("checkpoint %s: %s is %s %s, expected float64 %s"
                         % (path, os.path.basename(fn), xy.dtype, xy.shape, (model.batch, pm["count"], 2)))
    return xy


def from_checkpoint(cls, path, dist=None, **overrides):
    """``cls(**saved keywords, **overrides)`` restored from ``path`` (``Model.from_checkpoint``).  An override that gives
    the model a state slot the checkpoint lacks is refused by ``check``: YBJ and QL carry ``LAP2PHI`` only when
    ``nu4w != 0``, so their ``nu4w`` can change on restart between non-zero values or to zero, not from zero."""
    path = locate(path)
    meta = read_meta(path)
    if meta["model"] != _class_name(cls):
        raise ValueError("checkpoint %s holds a %s, not a %s" % (path, meta["model"], _class_name(cls)))
    changed = sorted(k for k, v in overrides.items() if k in meta["params"] and not _same(v, meta["params"][k]))
    if changed:
        warnings.warn("restarting %s with %s changed: the run does not continue the saved one exactly"
                      % (path, ", ".join("%s=%r (was %r)" % (k, overrides[k], meta["params"][k]) for k in changed)))
    kw = dict(meta["params"], **meta["run"])
    kw.update(nx=meta["nx"], batch=meta["batch"])
    kw.update(overrides)
    model = cls(**kw)
    load(model, path, dist=dist, changed=changed)
    return model
