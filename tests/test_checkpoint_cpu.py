"""The checkpoint file layer (niwqg_b200/Checkpoint.py) on CPU, with a stub device that holds its state in numpy arrays:
format round trip, the atomic replace, the version check, and the parallel writes and reads of a slab run (rows of the
physical slots, slab_kx columns of the spectral ones) over a world_size-2 gloo process group."""
import json
import os
import socket

import numpy as np
import pytest

from niwqg_b200 import Checkpoint as ck
from niwqg_b200 import _native as nat


class StubIO(object):
    """Device of one rank: this rank's rows / columns of every slot, as the native handle would return them."""

    def __init__(self, nx, batch, rank=0, nranks=1, dist=None, half=False):
        self.nx, self.batch, self.rank, self.nranks = nx, batch, rank, nranks
        self.half = half
        self.dist = dist
        self.state = {}
        self.carry = np.zeros(batch * 5)

    def slots(self):
        nk = self.nx // 2 + 1 if self.half else self.nx
        return [ck.Slot("QH", np.complex128, (self.nx, nk), "cols"), ck.Slot("PHI", np.complex128, (self.nx, self.nx), "rows"),
                ck.Slot("C", np.float64, (self.nx, self.nx), "rows")]

    def local(self, slot, whole):
        """This rank's part of a whole-grid array of one member."""
        return np.ascontiguousarray(whole[ck._local_index(slot, self)])

    def fill(self, glob):
        for s in self.slots():
            self.state[s.name] = np.stack([self.local(s, glob[s.name][m]) for m in range(self.batch)])

    def read(self, name, member):
        return self.state[name][member].copy()

    def write(self, name, member, a):
        self.state.setdefault(name, [None] * self.batch)[member] = np.array(a)

    def get_carry(self):
        return self.carry.copy()

    def set_carry(self, a):
        self.carry = np.array(a)

    def agree(self, ok):
        return ck.agree(self.dist, self.nranks, ok)


def _global_state(io, seed=7):
    rng = np.random.RandomState(seed)
    out = {}
    for s in io.slots():
        shape = (io.batch,) + s.shape
        a = rng.randn(*shape)
        out[s.name] = a + 1j * rng.randn(*shape) if s.dtype == np.complex128 else a
    return out


def _meta():
    return dict(model="test.Model", params={"dt": 0.1}, run={}, t=1.5, tc=3, status={})


@pytest.mark.parametrize("half", [False, True])
def test_format_round_trip(tmp_path, half):
    io = StubIO(16, 2, half=half)
    glob = _global_state(io)
    io.fill(glob)
    io.carry = np.arange(10.) / 3
    diags = {"Ke": np.array([1., 2.]), "time": np.array(0.5)}
    path = str(tmp_path / "ck")
    ck.write(path, _meta(), io, diags)
    meta = ck.read_meta(path)
    assert (meta["nx"], meta["batch"], meta["t"], meta["tc"]) == (16, 2, 1.5, 3)
    assert [s["name"] for s in meta["slots"]] == ["QH", "PHI", "C"]
    for s in io.slots():
        a = np.load(os.path.join(path, s.name + ".npy"))
        assert a.dtype == s.dtype and a.shape == (2,) + s.shape
        assert np.array_equal(a, glob[s.name])
    back = StubIO(16, 2, half=half)
    ck.check(path, meta, back)
    d = ck.read(path, meta, back)
    for s in io.slots():
        assert np.array_equal(np.stack(back.state[s.name]), glob[s.name])
    assert np.array_equal(back.carry, io.carry)
    assert set(d) == set(diags) and all(np.array_equal(d[k], diags[k]) for k in diags)
    assert not [f for f in os.listdir(str(tmp_path)) if f != "ck"]      # no temporary directory left behind


def test_failed_save_leaves_the_previous_checkpoint(tmp_path):
    io = StubIO(16, 1)
    glob = _global_state(io, 1)
    io.fill(glob)
    path = str(tmp_path / "ck")
    ck.write(path, _meta(), io)

    class Failing(StubIO):
        def read(self, name, member):
            if name == "PHI":
                raise IOError("device read failed")
            return StubIO.read(self, name, member)
    bad = Failing(16, 1)
    bad.fill(_global_state(bad, 2))
    with pytest.raises(IOError):
        ck.write(path, _meta(), bad)
    back = StubIO(16, 1)
    meta = ck.read_meta(path)
    ck.check(path, meta, back)
    ck.read(path, meta, back)
    for s in io.slots():
        assert np.array_equal(np.stack(back.state[s.name]), glob[s.name])
    # the next save replaces the old checkpoint and the leftover partial directory
    io2 = StubIO(16, 1)
    glob2 = _global_state(io2, 3)
    io2.fill(glob2)
    ck.write(path, _meta(), io2)
    assert os.listdir(str(tmp_path)) == ["ck"]
    assert np.array_equal(np.load(os.path.join(path, "PHI.npy")), glob2["PHI"])


def test_a_directory_that_is_not_a_checkpoint_is_never_replaced(tmp_path):
    io = StubIO(16, 1)
    io.fill(_global_state(io))
    data = tmp_path / "output"
    (data / "snapshots").mkdir(parents=True)
    (data / "snapshots" / "000.h5").write_bytes(b"snapshot")
    with pytest.raises(ValueError, match="not a checkpoint"):
        ck.write(str(data), _meta(), io)
    assert (data / "snapshots" / "000.h5").read_bytes() == b"snapshot"
    assert sorted(os.listdir(str(tmp_path))) == ["output"]       # nothing written beside it either
    (tmp_path / "afile").write_bytes(b"x")
    with pytest.raises(ValueError, match="not a checkpoint"):
        ck.write(str(tmp_path / "afile"), _meta(), io)
    (tmp_path / "empty").mkdir()
    ck.write(str(tmp_path / "empty"), _meta(), io)                # an empty directory is fine
    assert ck.read_meta(str(tmp_path / "empty"))["tc"] == 3


def test_an_interrupted_replacement_is_found_under_old(tmp_path):
    """A save that died between its two renames left the previous checkpoint under .<name>.old and none at <name>."""
    io = StubIO(16, 1)
    glob = _global_state(io)
    io.fill(glob)
    path = str(tmp_path / "ck")
    ck.write(path, _meta(), io)
    os.replace(path, str(tmp_path / ".ck.old"))
    with pytest.warns(UserWarning, match="interrupted save"):
        where = ck.locate(path)
    back = StubIO(16, 1)
    meta = ck.read_meta(where)
    ck.check(where, meta, back)
    ck.read(where, meta, back)
    assert np.array_equal(np.stack(back.state["PHI"]), glob["PHI"])
    io2 = StubIO(16, 1)
    io2.fill(_global_state(io2, 4))
    ck.write(path, _meta(), io2)                                   # the next save cleans up
    assert os.listdir(str(tmp_path)) == ["ck"] and ck.locate(path) == path


def test_version_and_missing_slot_are_refused(tmp_path):
    io = StubIO(16, 1)
    io.fill(_global_state(io))
    path = str(tmp_path / "ck")
    ck.write(path, _meta(), io)
    fn = os.path.join(path, ck.META)
    meta = json.load(open(fn))
    meta["version"] = ck.VERSION + 1
    json.dump(meta, open(fn, "w"))
    with pytest.raises(ValueError, match="version"):
        ck.read_meta(path)
    meta["version"] = ck.VERSION
    json.dump(meta, open(fn, "w"))
    os.remove(os.path.join(path, "C.npy"))
    back = StubIO(16, 1)
    with pytest.raises(FileNotFoundError, match="C.npy"):
        ck.check(path, ck.read_meta(path), back)
    with pytest.raises(ValueError, match="nx=16"):
        ck.check(path, ck.read_meta(path), StubIO(32, 1))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, path, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        N, B = 32, 2
        io = StubIO(N, B, rank, world, dist)
        glob = _global_state(io)
        io.fill(glob)
        io.carry = np.arange(B * 5.)
        ck.write(path, _meta(), io, {"Ke": np.array([1., 2.])})
        # read back on this layout: every rank gets exactly its own rows / columns
        back = StubIO(N, B, rank, world, dist)
        meta = ck.read_meta(path)
        ck.check(path, meta, back)
        ck.read(path, meta, back)
        ok = all(np.array_equal(np.stack(back.state[s.name]), io.state[s.name]) for s in io.slots())
        ok = ok and np.array_equal(back.carry, io.carry)
        # the columns this rank holds are the slab_kx columns of the natural-order spectrum
        ok = ok and np.array_equal(io.state["QH"][1], glob["QH"][1][:, nat.slab_kx(N, world, rank)])

        # a device read that fails on rank 1 only raises on both ranks (nobody waits for it at a barrier), and the
        # checkpoint written above stays as it was
        class Failing(StubIO):
            def read(self, name, member):
                if self.rank == 1 and name == "PHI":
                    raise IOError("device read failed")
                return StubIO.read(self, name, member)
        bad = Failing(N, B, rank, world, dist)
        bad.fill(_global_state(bad, 9))
        try:
            ck.write(path, _meta(), bad)
            ok = False
        except IOError:
            ok = ok and rank == 1
        except RuntimeError as e:
            ok = ok and rank == 0 and "another rank" in str(e)
        ok = ok and np.array_equal(np.load(os.path.join(path, "PHI.npy")), glob["PHI"])
        q.put((rank, ok))
    finally:
        dist.destroy_process_group()


def test_slab_writes_reassemble_natural_order_world2_gloo(tmp_path):
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    path = str(tmp_path / "ck")
    procs = [ctx.Process(target=_worker, args=(r, 2, port, path, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(ok for _, ok in res), res
    # the files hold the whole grid in natural order: a one-rank reader gets the global arrays
    io = StubIO(32, 2)
    glob = _global_state(io)
    meta = ck.read_meta(path)
    ck.check(path, meta, io)
    ck.read(path, meta, io)
    for s in io.slots():
        assert np.array_equal(np.stack(io.state[s.name]), glob[s.name]), s.name
