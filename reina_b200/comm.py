"""Process groups for the multi-GPU drivers, without any framework: one process per GPU, NCCL through the engine's own
C-ABI (include/reina_b200.h, rb_comm_*), and a file hand-off of the 128-byte NCCL unique id between the ranks of one
node.

A communicator object has `rank`, `size`, `allreduce(x, op='sum'|'max')`, `allgather(x)` and `barrier()`:

  * `LocalComm()`            one process: every call is the identity;
  * `EngineComm(engine)`     NCCL over NVLink through the engine handle (rb_comm_allreduce / rb_comm_allgather);
  * tests supply their own adapter over a CPU process group with the same five members (tests/helpers.py).

A communicator may also have `sendrecv({peer: bytes}) -> {peer: bytes}`, a collective in which every rank sends its
payloads and receives what the others sent it: ensemble.particle_filter moves replica records through it when the
communicator is not the engine's own EngineComm (which moves them device to device, rb_comm_move_replicas).

`connect(engine)` builds the right one from the launcher's environment (RANK / WORLD_SIZE, as torchrun sets them).
"""
import os
import tempfile
import time

import numpy as np

from . import _abi


def world():
    """(rank, world_size, local_rank) from the launcher's environment; (0, 1, 0) without one."""
    return (int(os.environ.get('RANK', '0')), int(os.environ.get('WORLD_SIZE', '1')),
            int(os.environ.get('LOCAL_RANK', '0')))


class LocalComm:
    rank, size = 0, 1

    def allreduce(self, x, op='sum'):
        return np.asarray(x, dtype=np.float64)

    def allgather(self, x):
        return np.asarray(x)[None]

    def barrier(self):
        pass


class EngineComm:
    """NCCL communicator joined through an engine handle (rb_comm_init or rb_shard_init)."""

    def __init__(self, engine):
        self.engine = engine
        f = engine.lib.f
        self.rank, self.size = f['comm_rank'](engine.h), f['comm_size'](engine.h)

    def allreduce(self, x, op='sum'):
        x = np.asarray(x, dtype=np.float64)
        return self.engine.comm_allreduce(x, op).reshape(x.shape)

    def allgather(self, x):
        return self.engine.comm_allgather(x)

    def barrier(self):
        self.engine.comm_allreduce(np.zeros(1))


_sequence = {}
_written = []


def _rendezvous_path(key):
    # the ranks of one launch share their parent (the launcher); MASTER_PORT tells concurrent launches apart
    tag = '%s_%s_%s' % (os.getppid(), os.environ.get('MASTER_PORT', '0'), key)
    return os.path.join(tempfile.gettempdir(), 'reina_b200_%s.uid' % tag)


def _cleanup():
    for p in _written:
        try:
            os.remove(p)
        except OSError:
            pass


def broadcast_bytes(payload, rank, key='comm', timeout=120.0):
    """Rank 0's `payload` (bytes) on every rank of this node's launch: written to a file under the temp directory
    (atomically, by rename), polled by the others.  Every rank must make the same sequence of calls: the n-th call for a
    key uses its own file, so an earlier hand-off is never read twice.  For several nodes hand the id over yourself."""
    seq = _sequence.get(key, 0)
    _sequence[key] = seq + 1
    path = _rendezvous_path('%s%d' % (key, seq))
    if rank == 0:
        tmp = path + '.tmp%d' % os.getpid()
        with open(tmp, 'wb') as f:
            f.write(payload)
        os.replace(tmp, path)
        if not _written:
            import atexit
            atexit.register(_cleanup)
        _written.append(path)
        return payload
    t0 = time.time()
    while True:
        try:
            with open(path, 'rb') as f:
                data = f.read()
            if data:
                return data
        except FileNotFoundError:
            pass
        if time.time() - t0 > timeout:
            raise _abi.EngineError('no unique id from rank 0 after %.0f s (%s)' % (timeout, path))
        time.sleep(0.01)


def connect(engine, rank=None, size=None, key='comm', unique_id=None):
    """Join `engine` to the NCCL communicator of this launch and return its EngineComm (LocalComm for one process)."""
    env_rank, env_size, _ = world()
    rank = env_rank if rank is None else rank
    size = env_size if size is None else size
    if size == 1:
        return LocalComm()
    if unique_id is None:
        unique_id = broadcast_bytes(_abi.shard_unique_id(engine.lib) if rank == 0 else None, rank, key)
    engine.comm_init(rank, size, unique_id)
    c = EngineComm(engine)
    c.barrier()
    return c
