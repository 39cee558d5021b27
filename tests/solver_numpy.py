"""Vectorised numpy restatement of the fused sync step for every solver (test infrastructure).

Written independently of oracle/sync_oracle.c and tests/solver_oracle.c, so that the C oracles are checked against
a second implementation: float32 arrays, one rounding per numpy operation (numpy does not contract a*x + y into an
FMA; np.sqrt and / on float32 are correctly rounded).
"""
import numpy as np

f32 = np.float32


def chunk(P, N, r):
    """socket_sync_cpu.cpp:46-54: multiply first, then divide."""
    lo, hi = r * P // N, (r + 1) * P // N
    return lo, hi - lo


def _update(g, w, h, h2, lr, ld, l1, type, m, delta, rms_decay):
    """Regularize + ComputeUpdateValue + Blob::Update of one blob (arrays are float32, updated in place)."""
    if ld != 0:
        x = ((f32(0) < w).astype(f32) - (w < f32(0)).astype(f32)) if l1 else w
        g = ld * x + g
    if type == "SGD":
        h[:] = m * h
        h[:] = lr * g + h
        g = h.copy()
    elif type == "Nesterov":
        u = h.copy()
        h[:] = m * h
        h[:] = lr * g + h
        u = (-m) * u
        u = (f32(1) + m) * h + u
        g = u
    elif type in ("AdaGrad", "RMSProp"):
        u = g * g
        if type == "AdaGrad":
            h[:] = u + h
        else:
            h[:] = rms_decay * h
            h[:] = (f32(1) - rms_decay) * u + h
        u = np.sqrt(h)
        u = u + delta
        u = g / u
        g = f32(0) * g
        g = lr * u + g
    elif type == "AdaDelta":
        u = g * g
        h[:] = m * h
        h[:] = (f32(1) - m) * u + h
        u = delta + h2
        t = delta + h
        u = u / t
        u = np.sqrt(u)
        g = g * u
        u = g * g
        h2[:] = m * h2
        h2[:] = (f32(1) - m) * u + h2
        g = lr * g
    else:
        raise ValueError(type)
    w[:] = f32(-1) * g + w


def step(data, diff, hist, hist2, counts, lr_mult, decay_mult, rate, momentum, weight_decay,
         regularization_type="L2", type="SGD", delta=1e-8, rms_decay=0.0):
    """One Solver::Step on len(data) ranks in place: all-gather, 1/N scale, ordered reduce-scatter, update."""
    N, P = len(data), data[0].size
    rate, m, wd = f32(rate), f32(momentum), f32(weight_decay)
    delta, rms_decay = f32(delta), f32(rms_decay)
    if N > 1:
        for owner in range(N):  # on_start: every rank takes the owner's shard
            o, s = chunk(P, N, owner)
            for r in range(N):
                data[r][o:o + s] = data[owner][o:o + s]
        inv = f32(1.0 / N)
        g = [inv * d for d in diff]
        for r in range(N):  # owner r adds r+1, r+2, ... (mod N) in that order: dst = recv + dst
            o, s = chunk(P, N, r)
            acc = g[r][o:o + s].copy()
            for k in range(1, N):
                acc = g[(r + k) % N][o:o + s] + acc
            diff[r][o:o + s] = acc
            for q in range(N):
                if q != r:
                    diff[q][o:o + s] = g[q][o:o + s]
    for r in range(N):
        b = 0
        for k, c in enumerate(counts):
            sl = slice(b, b + int(c))
            b += int(c)
            if c == 0:
                continue
            lr, ld = rate * f32(lr_mult[k]), wd * f32(decay_mult[k])
            _update(diff[r][sl].copy(), data[r][sl], hist[r][sl], hist2[r][sl] if hist2 is not None else None, lr, ld,
                    regularization_type == "L1", type, m, delta, rms_decay)
