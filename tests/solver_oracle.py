"""CPU oracle of the fused sync step with the Nesterov, AdaGrad, RMSProp and AdaDelta solvers (test infrastructure).

The sync half and SGD come from oracle/oracle.py (oracle/sync_oracle.c); the other solvers' ApplyUpdate is
tests/solver_oracle.c, compiled on first use into a temporary directory (the source tree may be read-only).
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
SOLVERS = ("SGD", "Nesterov", "AdaGrad", "RMSProp", "AdaDelta")
_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="cos_solver_oracle_")
        so = os.path.join(d, "libsolver_oracle.so")
        subprocess.run([os.environ.get("CC", "cc"), "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                        "-o", so, os.path.join(HERE, "solver_oracle.c"), "-lm"], check=True)
        L = ctypes.CDLL(so)
        pf, f32, i32, u64 = ctypes.POINTER(ctypes.c_float), ctypes.c_float, ctypes.c_int, ctypes.c_uint64
        L.cos_solver_oracle_apply_update.argtypes = [u64, u64, pf, pf, pf, pf, i32, ctypes.POINTER(ctypes.c_int64),
                                                     pf, pf, f32, f32, f32, i32, i32, f32, f32]
        _lib = L
    return _lib


def apply_update(begin, end, data, diff, hist, hist2, counts, lr_mult, decay_mult, rate, momentum, weight_decay,
                 regularization_type="L2", type="SGD", delta=1e-8, rms_decay=0.0):
    """SGDSolver::ApplyUpdate of solver `type` over elements [begin, end), in place (hist2: AdaDelta only)."""
    c, lm, dm = O._layout(counts, lr_mult, decay_mult)
    lib().cos_solver_oracle_apply_update(
        begin, end, O._pf(data), O._pf(diff), O._pf(hist), O._pf(hist2) if hist2 is not None else None, len(c),
        c.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), O._pf(lm), O._pf(dm), rate, momentum, weight_decay,
        int(regularization_type == "L1"), SOLVERS.index(type), delta, rms_decay)


def step(data, diff, hist, hist2, counts, lr_mult, decay_mult, rate, momentum, weight_decay,
         regularization_type="L2", type="SGD", delta=1e-8, rms_decay=0.0):
    """One Solver::Step on len(data) simulated ranks (in place), as cos_oracle_step_ex with solver `type`."""
    N, P = len(data), data[0].size
    if N > 1:
        O.all_gather(data)  # on_start
        for g in diff:
            O.scale(N, g)
        O.reduce_scatter(diff)
    for r in range(N):
        apply_update(0, P, data[r], diff[r], hist[r], hist2[r] if hist2 is not None else None, counts, lr_mult,
                     decay_mult, rate, momentum, weight_decay, regularization_type, type, delta, rms_decay)


class Simulation(O.Simulation):
    """oracle.Simulation with solver `type`; .hist2 holds AdaDelta's history of updates (None otherwise)."""

    def __init__(self, N, counts, lr_mult=None, decay_mult=None, type="SGD", delta=1e-8, rms_decay=0.0, **kw):
        super().__init__(N, counts, lr_mult, decay_mult, **kw)
        self.type, self.delta, self.rms_decay = type, delta, rms_decay
        self.hist2 = [np.zeros(self.P, np.float32) for _ in range(N)] if type == "AdaDelta" else None

    def step(self, grads=None):
        diff = grads if grads is not None else [self.gradient(r, self.iter) for r in range(self.N)]
        diff = [np.ascontiguousarray(g, dtype=np.float32).copy() for g in diff]
        rate = self.rate()
        step(self.data, diff, self.hist, self.hist2, self.counts, self.lr_mult, self.decay_mult, rate,
             self.hp["momentum"], self.hp["weight_decay"], self.regularization_type, self.type, self.delta,
             self.rms_decay)
        self.iter += 1
        return rate

    def consistent_history2(self):
        """AdaDelta's h2 as the shard owners hold it (None for the other solvers)."""
        if self.hist2 is None:
            return None
        out = np.empty(self.P, np.float32)
        for r in range(self.N):
            o, s = O.chunk(self.P, self.N, r)
            out[o:o + s] = self.hist2[r][o:o + s]
        return out
