"""The reference's own kernels as the GPU tests call them (the API of oracle/ref_ops.py), answered from stored outputs.

oracle/_ref/libref_ops.so is compiled from the original project's sources, which are not part of this repository, so
the tests do not run it.  tests/golden/ref_kernels/<test>.npz holds what it returned on a B200 for every call the test
makes, keyed by a digest of the call: operator, scalar arguments, and the dtype, shape and bytes of every input.  A
call whose inputs were never recorded fails.  To record (where oracle/_ref/libref_ops.so is built):

    python -m pytest tests -m gpu --record-ref-kernels DIR      then copy DIR/*.npz to tests/golden/ref_kernels/

TEST INFRASTRUCTURE ONLY.
"""
import hashlib
import os

import numpy as np
import torch


def _digest(op, args):
    h = hashlib.sha256(op.encode())
    for a in args:
        if isinstance(a, torch.Tensor):
            t = a.detach().contiguous().cpu()
            h.update(("%s%s" % (t.dtype, tuple(t.shape))).encode())
            h.update(t.numpy().tobytes())
        else:
            h.update(float(a).hex().encode())
    return h.hexdigest()[:32]


class Stored:
    """Replays the outputs stored in one .npz file (entries <digest>_<output number>)."""

    def __init__(self, path):
        self.path = path
        self.arrays = np.load(path) if os.path.exists(path) else {}

    def __getattr__(self, op):
        def call(*args):
            key = _digest(op, args)
            dev = next(a.device for a in args if isinstance(a, torch.Tensor))
            outs = []
            while "%s_%d" % (key, len(outs)) in self.arrays:
                outs.append(torch.from_numpy(self.arrays["%s_%d" % (key, len(outs))]).to(dev))
            if not outs:
                raise AssertionError("%s holds no output of the reference's %s for these inputs: record them again "
                                     "(oracle/ref_golden.py)" % (self.path, op))
            return outs[0] if len(outs) == 1 else tuple(outs)
        return call


class Recording:
    """Runs the live kernels (oracle.ref_ops) and keeps every call's outputs in `store` for write()."""

    def __init__(self, live, store):
        self.live, self.store = live, store

    def __getattr__(self, op):
        fn = getattr(self.live, op)

        def call(*args):
            key = _digest(op, args)
            out = fn(*args)
            for j, o in enumerate(out if isinstance(out, tuple) else (out,)):
                self.store["%s_%d" % (key, j)] = o.cpu().numpy()
            return out
        return call


def write(recordings, out_dir):
    """recordings: {test name: store of a Recording} -> out_dir/<test name>.npz."""
    os.makedirs(out_dir, exist_ok=True)
    for name, store in recordings.items():
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), **store)
