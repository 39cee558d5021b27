"""Kernel time of the fused sync step per solver (SGD as the control), on the GPU:
   python scripts/bench_solvers.py [--iters 50] [--out profiles/r03_bench_solvers.json]

Each row times one sync_step launch with CUDA events on the net's stream (option "timing"), median over --iters
launches after 5 warm-up launches; the gradient is refilled before every launch, outside the timed window.  No L2
flush: at CaffeNet size every buffer (244 MB) is larger than the 126 MB L2, so each launch streams from HBM.
Rows whose GPU count the machine does not have are written with "not measured"."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SOLVERS = {  # the reference's example hyper-parameters; momentum 0 where the solver forbids it
    "SGD": dict(momentum=0.9),
    "Nesterov": dict(momentum=0.95),
    "AdaGrad": dict(momentum=0.0, delta=1e-8),
    "RMSProp": dict(momentum=0.0, rms_decay=0.98, delta=1e-8),
    "AdaDelta": dict(momentum=0.95, delta=1e-6),
}
CASES = [("caffenet", 1, None), ("caffenet", 2, 2), ("caffenet", 8, 2), ("lenet", 2, 4)]  # (net, N, forced kernel)
COPY_PEAK = 6585e9  # B/s, measured device-to-device copy peak of this B200 (DESIGN.md §5)


def algorithmic_bytes(solver, P):
    """HBM bytes of one N = 1 launch: read g, w, h and write w, h and g = 0 (6 x 4P), plus AdaDelta's h2 read and
    write (2 x 4P)."""
    return (32 if solver == "AdaDelta" else 24) * P


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def time_case(cos, net_name, N, kernel, solver, iters):
    import numpy as np
    import torch
    from caffeonspark_b200 import nets
    from gpu_util import Ranks
    desc = nets.solver_desc(net_name, type=solver, **SOLVERS[solver])
    opts = dict(timing=1)
    if kernel is not None:
        opts["kernel"] = kernel
    R = Ranks(cos, desc, N, devices=list(range(N)), timeout_ms=20000, **opts)
    try:
        for r, net in enumerate(R.nets):
            net.fill("data", 1, 0, 0.05)
        R.connect()
        resolved = R.nets[0].get_option("resolved_kernel")
        ms = []
        for t in range(iters + 5):
            for r, net in enumerate(R.nets):
                net.fill("diff", 1, (t + 1) * 4096 + r, 0.01)
            for net in R.nets:
                assert net.sync_step(0), net.last_error()
            for net in R.nets:
                assert net.synchronize(), net.last_error()
            if t >= 5:
                ms.append(max(net.last_kernel_ms() for net in R.nets))
        torch.cuda.synchronize()
        return dict(us_median=float(np.median(ms)) * 1e3, us_min=float(np.min(ms)) * 1e3, resolved_kernel=resolved,
                    P=desc.param_count)
    finally:
        R.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import caffeonspark_b200 as cos
    ngpu = torch.cuda.device_count()
    if ngpu == 0:
        raise SystemExit("bench_solvers.py needs a GPU")
    rows = []
    for net_name, N, kernel in CASES:
        for solver in SOLVERS:
            row = dict(net=net_name, N=N, solver=solver)
            if N > ngpu:
                row["result"] = "not measured"
            else:
                row.update(time_case(cos, net_name, N, kernel, solver, a.iters))
                if N == 1:
                    b = algorithmic_bytes(solver, row["P"])
                    row["algorithmic_bytes"] = b
                    row["hbm_GBps"] = b / (row["us_median"] * 1e-6) / 1e9
                    row["share_of_copy_peak"] = b / COPY_PEAK / (row["us_median"] * 1e-6)
            rows.append(row)
            print(json.dumps(row), flush=True)
    out = dict(gpu=gpu_info(), gpus=ngpu, iters=a.iters,
               timing="CUDA events around each launch on the net's stream, median; no L2 flush (buffers > L2)",
               rows=rows)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(dict(gpu=out["gpu"], gpus=ngpu)))


if __name__ == "__main__":
    main()
