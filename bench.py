#!/usr/bin/env python
"""bench.py -- images/sec of synchronous data-parallel SGD with the B200-native
gradient-sync library, next to the reference's CPU socket path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload lenet|cifar10_quick|caffenet]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
         --master-port P bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...     # the reference's own CPU sync path (oracle/_ref)
  python bench.py --sweep --gpus N         # config 5: all-reduce message-size sweep

A "step" is one Solver::Step: Net::ForwardBackward (PyTorch/cuDNN harness, NOT
part of the product) followed by the hot path -- ONE launch of the fused
scale + reduce-scatter + SGD/momentum + weight all-gather kernel.
 value  : inputs resident in HBM, device-timed (CUDA events per step, summed;
          max over ranks), L2 flushed between steps outside the timed events.
 e2e    : the reference-facing call CaffeNet.train(0, FloatBlob[]) with pinned
          HOST blobs: H2D of the batch and D2H of the loss inside the timed region.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# Rank 0 prints exactly ONE JSON line on stdout.  Native libraries write to file descriptor 1 behind
# Python's back (NCCL prints its "NCCL version ..." banner there at every debug level >= VERSION), so the
# real stdout is set aside and fd 1 points at stderr for the whole run; emit() writes the line to the saved fd.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)
sys.stdout = sys.stderr


def emit(obj):
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


NVLINK_MEASURED_GBS = 770.0  # B200_PROFILING.md: measured peer copy per direction (900 nominal)
HBM_FALLBACK_GBS = 6650.0    # B200_PROFILING.md fallback if MEASURED_PEAKS.json is absent


def env_int(name, default):
    return int(os.environ.get(name, default))


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": HBM_FALLBACK_GBS}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.rows, self.proc, self.device = [], None, device

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i] == "Active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cuda_time_steps(torch, dist, world, steps, warmup, step_fn, flush_fn, before_last=None):
    """W warm-up steps, then K steps each bracketed by CUDA events on the
    current stream (L2 flush between steps, outside the events; before_last,
    if given, runs outside the events ahead of the last step); barrier +
    synchronize on both sides; returns max-over-ranks total ms."""
    for _ in range(warmup):
        step_fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i, (a, b) in enumerate(evs):
        if before_last is not None and i == steps - 1:
            before_last()
        flush_fn()
        a.record()
        step_fn()
        b.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    total = sum(a.elapsed_time(b) for a, b in evs)
    if world > 1:
        t = torch.tensor([total], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total = float(t.item())
    return total


DUMP_MAX_ELEMS = 1 << 22  # per array: 16 MiB of float32, so the dump of all three workloads stays under 64 MiB


def dump_outputs(torch, out_dir, prefix, arrays):
    """Writes each device array as <out_dir>/<prefix>_<key>.npy in float32.  An array longer than DUMP_MAX_ELEMS is
    replaced by a fixed sample: one element out of every stretch of n // DUMP_MAX_ELEMS, at an offset drawn from a
    generator seeded with n, so every run writes the same positions."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for key, t in arrays.items():
        t = t.detach().reshape(-1).float()
        n = t.numel()
        if n > DUMP_MAX_ELEMS:
            stride = n // DUMP_MAX_ELEMS
            idx = np.arange(DUMP_MAX_ELEMS, dtype=np.int64) * stride + \
                np.random.default_rng(n).integers(0, stride, DUMP_MAX_ELEMS)
            t = t[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, f"{prefix}_{key}.npy"), t.cpu().numpy().astype(np.float32))


def algorithmic_bytes(P, world, mode, zero_diff, bf16, nvls=False, push=False):
    """DESIGN.md section 'algorithmic bytes': per launch, per GPU.
    -> (hbm_bytes, nvlink_bytes_per_direction)"""
    z = 4 * P if zero_diff else 0
    if world == 1:
        return 20 * P + z, 0                      # read g,w,h ; write w,h (+ zero g)
    bg = 2 if bf16 else 4
    f = (world - 1) / world
    if nvls:                                      # switch reads every rank once, owner multicasts its shard
        hbm = 4 * P + 4 * P + 12 * P / world + z  # serve the switch's reads, land the multicast, own w/h
        return hbm, 4 * P * (1 + 1 / world)       # up: 4P served + 4P/N stored; down: 4P/N reduced + 4P landed
    if push:                                      # cast in registers: no wire buffer; slots written + read once
        hbm = 4 * P + 2 * bg * P * f + 4 * P * f + 16 * P / world + z
        return hbm, (bg + 4) * P * f
    cast = (4 * P + 2 * P) if bf16 else 0         # pull kernels, phase 0: read fp32, write bf16 wire
    if mode == 2:                                 # one-shot: read all peers' full gradient, update everything
        return cast + bg * P + 20 * P + z, bg * P * (world - 1)
    hbm = cast + bg * P + 4 * P * f + 12 * P / world + 4 * P / world + z  # serve grads, land pushes, own shard
    return hbm, (bg + 4) * P * f                  # pull grads + push weights


class NvlinkCounters:
    """NVML per-GPU NVLink data counters (KiB, summed over the links): payload bytes that really crossed the
    links, read before/after K launches -- evidence that is not events / formula."""
    IDS = {"data_tx": 138, "data_rx": 139, "raw_tx": 140, "raw_rx": 141}  # NVML_FI_DEV_NVLINK_THROUGHPUT_*

    def __init__(self, torch, device):
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            uuid = str(torch.cuda.get_device_properties(device).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
        except Exception as e:  # no NVML / no NVLink: the caller reports traffic as unavailable
            self.err = repr(e)

    def read(self):
        if self.h is None:
            return None
        try:
            vals = self.nv.nvmlDeviceGetFieldValues(self.h, [(i, 0xFFFFFFFF) for i in self.IDS.values()])
            out = {}
            for k, v in zip(self.IDS, vals):
                if v.nvmlReturn != 0:
                    return None
                out[k] = int(v.value.ullVal) * 1024
            return out
        except Exception:
            return None


def measure_nvlink_traffic(torch, dist, net, world, launches=50):
    """NVLink payload bytes per fused-kernel launch on this rank's GPU (NVML counters around `launches`
    back-to-back launches; the counters tick in KiB, so many launches are needed for small nets)."""
    ctr = NvlinkCounters(torch, torch.cuda.current_device())
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    c0 = ctr.read()
    with torch.cuda.stream(st):
        for _ in range(launches):
            if not net.sync_step(0, st.cuda_stream):
                raise RuntimeError(net.last_error())
    torch.cuda.synchronize()
    if not net.synchronize():
        raise RuntimeError(net.last_error())
    if world > 1:
        dist.barrier()
    time.sleep(0.05)
    c1 = ctr.read()
    if c0 is None or c1 is None:
        return None
    return {k: (c1[k] - c0[k]) / launches for k in c0}


def parity_check(torch, dist, C, harness, desc, name, rank, world, local, args, kernels):
    """Outside every timed region: two seeded steps on fresh nets, on ALL ranks, compared with the CPU oracle on
    rank 0 (this is the `cpu_baseline` leg, the one place bench.py may use oracle/).  Weights / gradients come
    from the device-side generator that is bit-identical to cos_oracle_fill.  Every rank must hold identical
    bits; rank 0's full weights and own history shard are compared with oracle.Simulation element by element
    (bit-exact for the P2P kernels; the NVLS kernel is held to the north star's 1e-5 relative)."""
    import numpy as np
    seed, res = 20260921, {}
    expected = None
    for kern in kernels:
        cl = harness.Cluster(desc, rank=rank, world=world, device=local)
        net = cl.net
        net.set_option("kernel", kern)
        net.set_option("nvls", int(args.nvls) if kern in (-1, 3) else 0)
        net.set_option("barrier_timeout_ms", 120000)
        net.fill("data", seed, 0, 0.05)
        torch.cuda.synchronize()
        cl.start()
        for t in range(2):
            net.fill("diff", seed, (t + 1) * 4096 + rank, 0.01)
            if not (net.sync_step(0) and net.synchronize()):
                raise RuntimeError(net.last_error())
        w = net.data()
        o, n = net.shard()
        sums = torch.stack([w.view(torch.int32).to(torch.int64).sum(), (w.view(torch.int32).to(torch.int64) *
                            torch.arange(1, w.numel() + 1, device=w.device, dtype=torch.int64) % 1000003).sum()])
        if world > 1:
            allsums = [torch.zeros_like(sums) for _ in range(world)]
            dist.all_gather(allsums, sums)
            same = all(bool((a == allsums[0]).all()) for a in allsums)
        else:
            same = True
        kname = KERNEL_NAMES[int(net.get_option("resolved_kernel"))]
        entry = {"kernel": kname, "nvls_active": bool(net.get_option("nvls_active")), "all_ranks_identical": same}
        if rank == 0:
            from oracle import oracle as O
            if expected is None:
                sim = O.Simulation(world, desc.counts, desc.lr_mult, desc.decay_mult, seed=seed,
                                   bf16=(desc.grad_dtype == "bf16"), **desc.hyper())
                sim.step()
                sim.step()
                expected = (sim.consistent_weights(), sim.consistent_history())
                del sim
            gw = w.cpu().numpy()
            gh = net.history()[o:o + n].cpu().numpy()
            ew, eh = expected[0], expected[1][o:o + n]
            bit = bool(np.array_equal(gw.view(np.uint32), ew.view(np.uint32)) and
                       np.array_equal(gh.view(np.uint32), eh.view(np.uint32)))
            big = np.abs(ew) > 1e-3 * float(np.max(np.abs(ew)))  # relative error where the weight is not ~0
            entry.update({"bit_exact": bit, "max_abs_err_weights": float(np.max(np.abs(gw - ew))),
                          "max_abs_weight": float(np.max(np.abs(ew))),
                          "max_rel_err_weights": float(np.max(np.abs(gw - ew)[big] / np.abs(ew)[big])) if big.any() else 0.0,
                          "max_abs_err_history": float(np.max(np.abs(gh - eh))) if n else 0.0,
                          "within_1e-5": bool(np.allclose(gw, ew, rtol=1e-5, atol=1e-8) and
                                              np.allclose(gh, eh, rtol=1e-5, atol=1e-9))})
        res[kname] = entry
        if not net.sync():
            raise RuntimeError(net.last_error())
        net.deallocate()
        if world > 1:
            dist.barrier()
    return res


def measure_workload(torch, dist, C, harness, nets, args, name, grad_dtype, rank, world, local, primary):
    """One workload, one net: device-resident `value`, host-blob `e2e`, in-step kernel time + roofline."""
    bf16 = grad_dtype == "bf16"
    desc = nets.solver_desc(name, grad_dtype=grad_dtype)
    batch = nets.NETS[name]["batch"]
    cl = harness.Cluster(desc, rank=rank, world=world, device=local)
    net = cl.net
    if args.algo:
        net.set_option("algo", args.algo)
    net.set_option("kernel", args.kernel)
    net.set_option("nvls", int(args.nvls))
    net.set_option("barrier_timeout_ms", 60000)
    prod = harness.make_producer(name, net)
    cl.start()
    P = net.param_count()
    w0 = net.data().clone() if args.dump_outputs else None
    mode = int(net.get_option("resolved_algo"))
    zero = int(net.get_option("zero_diff"))
    kern = int(net.get_option("resolved_kernel"))
    nvls = bool(net.get_option("nvls_active")) and kern == 3

    # synthetic batch: uniform[0,1) images, random labels; different per rank
    g = torch.Generator().manual_seed(1 + rank)
    c, h, w = nets.NETS[name]["input"]
    x_host = torch.rand((batch, c, h, w), generator=g).pin_memory()
    y_host = torch.randint(0, nets.NETS[name]["classes"], (batch, 1, 1, 1), generator=g).float().pin_memory()
    x_dev, y_dev = x_host.cuda(non_blocking=True), y_host.cuda().view(-1).long()
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    working_set = 3 * 4 * P
    need_flush = working_set < (256 << 20)

    def flush():
        if need_flush:
            flush_buf.zero_()

    # Everything below runs on ONE explicit stream.  (torch's default stream has the handle 0, which the
    # C ABI reads as "use the net's own stream": forward/backward and the sync launch would then sit on
    # two unordered streams and the sync kernel would fall outside the timed events.)
    work = torch.cuda.Stream()
    work.wait_stream(torch.cuda.current_stream())
    torch.cuda.set_stream(work)
    assert torch.cuda.current_stream().cuda_stream != 0

    # Net::ForwardBackward, captured in a CUDA graph when possible (launch-bound for the small nets)
    graph = None
    last = {}  # the loss of the latest forward/backward
    if not args.no_graph:
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    prod.forward_backward(x_dev, y_dev)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                last["loss"] = prod.forward_backward(x_dev, y_dev)
            net.diff().zero_()
        except Exception as e:  # eager fallback for the producer only (not the product path)
            graph = None
            if rank == 0:
                print(f"[bench] CUDA-graph capture of the gradient producer failed ({e}); eager", file=sys.stderr)
            net.diff().zero_()
    torch.cuda.synchronize()

    def fb():
        if graph is not None:
            graph.replay()
        else:
            last["loss"] = prod.forward_backward(x_dev, y_dev)

    def step():
        fb()
        if not net.sync_step(0, torch.cuda.current_stream().cuda_stream):
            raise RuntimeError(net.last_error())

    sampler = ClockSampler(local)
    if rank == 0 and primary:
        sampler.start()
    t_end = time.perf_counter() + (0.4 if primary else 0.0)  # nvidia-smi needs a moment to emit its first rows
    spin = torch.tensor([1], device="cuda")
    while True:                        # collective: every rank runs the same number of extra steps
        for _ in range(10):
            step()
        spin[0] = 1 if time.perf_counter() < t_end else 0
        if world > 1:
            dist.all_reduce(spin, op=dist.ReduceOp.MIN)
        if int(spin.item()) == 0:
            break
    torch.cuda.synchronize()

    def restart():
        # --dump-outputs: how many steps ran before the last timed one depends on the clock (the loop above), so
        # that step starts from the initial weights, zero history, iteration 0 and a reseeded dropout generator:
        # its outputs are then the same from run to run
        net.data().copy_(w0)
        net.history().zero_()
        net.diff().zero_()
        net.set_option("iter", 0)
        torch.cuda.manual_seed(1234)

    launches0 = net.launch_count()
    total_ms = cuda_time_steps(torch, dist, world, args.steps, args.warmup, step, flush,
                               before_last=restart if args.dump_outputs else None)
    launches = net.launch_count() - launches0 - args.warmup
    if not net.synchronize():
        raise RuntimeError(net.last_error())
    if args.dump_outputs and rank == 0:
        o, n = net.shard() if world > 1 else (0, P)  # history is kept on the owner of each shard
        dump_outputs(torch, args.dump_outputs, name + ("_bf16" if bf16 else ""),
                     {"weights": net.data(), "history": net.history()[o:o + n], "loss": last["loss"]})

    # The fused kernel IN the step: library-side CUDA events around the one launch, on the launching stream,
    # with forward/backward queued right in front of it (so the ranks arrive as they do in training: skewed by
    # their own forward/backward times, gradients partly still in L2).  L2 flushed before each forward/backward.
    net.set_option("timing", 1)
    kms = []
    for _ in range(max(5, min(args.steps, 30))):
        flush()
        step()
        kms.append(net.last_kernel_ms())  # waits for the launch
    net.set_option("timing", 0)
    k_ms = k_min_rank = sorted(kms)[len(kms) // 2]
    if world > 1:
        t = torch.tensor([k_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        k_ms = float(t.item())
        # the rank that arrives LAST never waits for a peer's forward/backward: its time is the kernel's own cost
        t = torch.tensor([k_min_rank], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        k_min_rank = float(t.item())
    # and back to back (no forward/backward in between, all ranks in lock step): K launches / K
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    net.sync_step(0, torch.cuda.current_stream().cuda_stream)
    ea.record()
    for _ in range(20):
        net.sync_step(0, torch.cuda.current_stream().cuda_stream)
    eb.record()
    torch.cuda.synchronize()
    k_b2b = ea.elapsed_time(eb) / 20
    if world > 1:
        t = torch.tensor([k_b2b], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        k_b2b = float(t.item())
    # forward/backward alone (reported so the split is visible)
    fb_evs = []
    for _ in range(10):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fb()
        b.record()
        fb_evs.append((a, b))
    torch.cuda.synchronize()
    fb_ms = sorted(a.elapsed_time(b) for a, b in fb_evs)[5]
    net.diff().zero_()
    torch.cuda.synchronize()

    # end to end through the reference-facing API: train(solver_index, host blobs).  train() double-buffers the
    # input staging (H2D of batch t+1 overlaps step t) and reads the loss back every step; the timed region ends
    # with synchronize(), i.e. when the last step's weights and loss are complete.
    for _ in range(max(args.warmup, 10)):  # both staging sets reach the producer's CUDA-graph replay (4 calls each)
        assert net.train(0, [x_host, y_host]), net.last_error()
    assert net.synchronize(), net.last_error()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e2e_launch0 = net.launch_count()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        if not net.train(0, [x_host, y_host]):
            raise RuntimeError(net.last_error())
    if not net.synchronize():
        raise RuntimeError(net.last_error())
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_launches = net.launch_count() - e2e_launch0
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    last_loss = net.last_loss()
    clocks = sampler.stop() if (rank == 0 and primary) else None

    peaks, peak_kind = measured_peaks()
    hbm_b, nvl_b = algorithmic_bytes(P, world, mode, zero, bf16, nvls=nvls, push=(kern in (2, 4)))
    if world == 1:
        bound, alg, peak = "hbm", hbm_b, float(peaks["hbm_gbs"])
    else:
        bound, alg, peak = "nvlink", nvl_b, NVLINK_MEASURED_GBS
    achieved = alg / (k_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    if world == 1:
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                traffic = json.load(f).get(f"{name}_n{world}")
            traffic_src = "ncu --set full dram__bytes_read.sum + dram__bytes_write.sum per launch (profiles/traffic.json)"
        except Exception:
            pass
    else:
        tr = measure_nvlink_traffic(torch, dist, net, world, launches=50 if P > (1 << 22) else 400)
        if tr is not None:
            traffic = max(tr["data_tx"], tr["data_rx"])
            traffic_src = ("NVML NVLink payload counters of this GPU around back-to-back launches, per launch: "
                           f"tx {tr['data_tx']:.0f} B, rx {tr['data_rx']:.0f} B (raw incl. protocol: tx "
                           f"{tr['raw_tx']:.0f} B, rx {tr['raw_rx']:.0f} B)")
    kernel_fn = {0: "fused_sync_sgd_kernel", 1: "fused_sync_sgd_tma_kernel", 2: "fused_sync_sgd_push_kernel",
                 3: "fused_sync_sgd_nvls_kernel", 4: "fused_sync_sgd_ll_kernel"}[kern]
    out = {
        "value": world * batch * args.steps / (total_ms * 1e-3), "unit": "images/s",
        "ms_per_step": total_ms / args.steps,
        "dtype": "f32" if not bf16 else "f32 (bf16 gradient wire)",
        "config": {"workload": f"{name} (batch {batch}/device, P={P} fp32 params), synchronous SGD: "
                               f"forward/backward + gradient sync + SGD update",
                   "global_batch": world * batch, "parallelism": f"dp{world}"},
        "impl_config": {"algo": {0: "local", 1: "two_shot", 2: "one_shot"}[mode], "grad_dtype": grad_dtype,
                        "kernel": KERNEL_NAMES[kern], "nvls": nvls,
                        "producer": "PyTorch/cuDNN forward/backward, " + ("cuda_graph" if graph is not None else "eager"),
                        "l2": "flushed between steps (256 MiB write outside the timed events)" if need_flush
                              else f"working set {working_set >> 20} MiB > 126 MiB L2"},
        "e2e": {"value": world * batch * args.steps / e2e_s, "unit": "images/s",
                "h2d_bytes_per_step": int(x_host.numel() * 4 + y_host.numel() * 4), "d2h_bytes_per_step": 4,
                "timing": "host wall clock around K train() calls + the final synchronize(); train() stages the "
                          "batch from pinned host memory on a copy stream (double buffered) and reads the loss "
                          "back every step; max over ranks", "last_loss": last_loss},
        "gpu_launches": int(launches), "e2e_gpu_launches": int(e2e_launches),
        "roofline": {"bound": bound, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "kernel": kernel_fn, "kernel_ms": k_ms,
                     "kernel_ms_how": "median of CUDA-event times around the launch inside full steps, max over ranks "
                                      "(includes waiting for the slowest rank's forward/backward)",
                     "kernel_ms_min_over_ranks": k_min_rank, "kernel_ms_back_to_back": k_b2b,
                     "algorithmic_bytes": alg, "peak_source": (peak_kind + " MEASURED_PEAKS.json hbm_gbs") if
                     world == 1 else "B200_PROFILING.md measured peer copy per direction"},
        "split_ms": {"forward_backward": fb_ms, "fused_sync_kernel": k_ms},
    }
    if clocks is not None:
        out["clocks"] = clocks
    if world > 1:
        out["bus_gbs"] = 4 * P * 2 * (world - 1) / world / (k_ms * 1e-3) / 1e9
        # the library route the fused kernel replaces: NCCL all-reduce of the fp32 gradient (the SGD update
        # would still need a separate >= 20P-byte elementwise pass on top of this)
        buf = torch.zeros(P, device="cuda")
        nc = []
        for i in range(13):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dist.barrier()
            a.record()
            dist.all_reduce(buf)
            b.record()
            torch.cuda.synchronize()
            if i >= 3:
                nc.append(a.elapsed_time(b))
        t = torch.tensor([sorted(nc)[len(nc) // 2]], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out["nccl_allreduce_only_ms"] = float(t.item())
        del buf
    if rank == 0 and world == 1 and primary and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(name, desc, batch, 1, fb_ms)
    net.deallocate()
    del prod, graph
    torch.cuda.set_stream(torch.cuda.default_stream())
    if world > 1:
        dist.barrier()
    return out, desc


def run_ours(args):
    import torch
    import torch.distributed as dist
    import caffeonspark_b200 as C
    from caffeonspark_b200 import harness, nets

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.backends.cudnn.benchmark = not os.environ.get("COS_BENCH_NO_AUTOTUNE")  # off under ncu launch lists
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True

    main, desc = measure_workload(torch, dist, C, harness, nets, args, args.workload, args.grad_dtype, rank, world,
                                  local, primary=True)
    out = {"metric": "images/sec", "value": main["value"], "unit": "images/s", "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "data": "synthetic"}
    out.update({k: v for k, v in main.items() if k not in ("value", "unit", "ms_per_step")})
    # the other BASELINE configs as extra keys, each with its own roofline (config 2: LeNet; config 3:
    # CIFAR-10-quick with the bf16 gradient wire)
    if args.extras:
        out["workloads"] = {}
        for wname, gd in (("lenet", "fp32"), ("cifar10_quick", "bf16")):
            if (wname, gd) == (args.workload, args.grad_dtype):
                continue
            r, _ = measure_workload(torch, dist, C, harness, nets, args, wname, gd, rank, world, local, primary=False)
            out["workloads"][wname + ("_bf16" if gd == "bf16" else "")] = r
    if world > 1 and not args.no_parity:
        # what ran in the timed region (AUTO) and, when that is the NVLS kernel, the bit-exact P2P kernel too
        kernels = [args.kernel]
        if main["impl_config"]["kernel"] == KERNEL_NAMES[3]:
            kernels.append(1)
        par = parity_check(torch, dist, C, harness, desc, args.workload, rank, world, local, args, kernels)
        out["parity"] = {"checked": True, "steps": 2, "against": "oracle.Simulation (C restatement pinned to the "
                         "reference's socket_sync_cpu.cpp) on rank 0's host", "kernels": par,
                         "bit_exact": all(v.get("bit_exact", False) for v in par.values() if not v["nvls_active"]) if
                         rank == 0 else None,
                         "all_within_1e-5": all(v.get("within_1e-5", False) for v in par.values()) if rank == 0 else None}
    if rank == 0 and args.kernels:
        out["kernel_rooflines"] = kernel_rooflines(C, nets, measured_peaks()[0], world, args.kernel)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(out)


def kernel_rooflines(C, nets, peaks, world, kernel=-1):
    """Fused-kernel-only timing of the three BASELINE layouts at N=1 (HBM roofline)."""
    import torch
    res = {}
    if world != 1:
        return res
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for name in ("lenet", "cifar10_quick", "caffenet"):
        desc = nets.solver_desc(name)
        net = C.CaffeNet(desc, "", "", 1, 1, 0, True, 0, torch.cuda.current_device() - 1, 0)
        net.connect([])
        net.set_option("kernel", kernel)
        net.set_option("timing", 1)
        P = net.param_count()
        net.diff().normal_(0, 0.01)
        ms = []
        for i in range(25):
            flush_buf.zero_()
            torch.cuda.synchronize()
            net.sync_step(0)
            net.synchronize()
            if i >= 5:
                ms.append(net.last_kernel_ms())
        k = sorted(ms)[len(ms) // 2]
        alg = 24 * P
        res[name] = {"P": P, "kernel_ms": k, "achieved_gbs": alg / (k * 1e-3) / 1e9,
                     "frac_of_hbm_peak": alg / (k * 1e-3) / 1e9 / float(peaks["hbm_gbs"]), "algorithmic_bytes": alg}
        net.deallocate()
    return res


def cpu_baseline(name, desc, batch, world, fb_ms):
    """The reference's CPU sync path on this box's host cores, bounded sample."""
    from oracle import oracle as O
    P = desc.param_count
    cores = os.cpu_count()
    # ~10-20 s of CPU work: measured rates are ~0.4 GB/s (socket path) / ~2 GB/s (local update)
    if O.ref_available():
        est_ms = max(0.5, 4 * P / 1e6 * (4.0 if world > 1 else 1.0) * world)
        iters = int(max(4, min(2000, 10000 / est_ms)))  # ~10 s of CPU work, bounded
        r = O.run_ref_time(world, desc.counts, desc.lr_mult, desc.decay_mult, iters=iters, **desc.hyper())
        sync_ms, kind = r["ms_per_iter_median"], "reference"
        used = world  # one solver thread per executor process (+ its receiver threads)
    else:
        import numpy as np
        sim = O.Simulation(world, desc.counts, desc.lr_mult, desc.decay_mult, **desc.hyper())
        grads = [sim.gradient(r, 0) for r in range(world)]
        iters = 5
        t0 = time.perf_counter()
        for _ in range(iters):
            sim.step(grads)
        sync_ms, kind, used = (time.perf_counter() - t0) * 1e3 / iters, "port", 1
        del np
    return {"value": world * batch / ((sync_ms + fb_ms) * 1e-3), "unit": "images/s", "cores": used,
            "host_cores": cores, "kind": kind,
            "sample": f"{iters} iterations of the reference's CPU sync+update at P={P}, N={world} "
                      f"(median {sync_ms:.3f} ms/iter, first dropped) + the same GPU forward/backward time "
                      f"({fb_ms:.3f} ms) as this run, so only the sync differs",
            "sync_ms_per_iter": sync_ms}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path
    (oracle/_ref = socket.cpp + socket_sync_cpu.cpp + parallel_cpu.cpp compiled
    verbatim, N loopback processes) + the PyTorch forward/backward time."""
    rank, world = env_int("RANK", 0), env_int("WORLD_SIZE", 1)
    if rank != 0:
        return
    world = max(world, args.gpus)
    import torch
    from caffeonspark_b200 import nets
    name = args.workload
    desc = nets.solver_desc(name)
    batch = nets.NETS[name]["batch"]
    fb_ms = 0.0
    if torch.cuda.is_available():
        torch.backends.cudnn.benchmark = True
        torch.backends.cuda.matmul.allow_tf32 = True
        torch.backends.cudnn.allow_tf32 = True
        mod = nets.torch_module(name).cuda()
        for prm in mod.parameters():
            prm.grad = torch.zeros_like(prm)
        c, h, w = nets.NETS[name]["input"]
        x = torch.rand((batch, c, h, w), device="cuda")
        y = torch.randint(0, nets.NETS[name]["classes"], (batch,), device="cuda")
        lossf = torch.nn.CrossEntropyLoss()

        def fb():
            lossf(mod(x), y).backward()

        # same forward/backward execution as our arm (CUDA-graph replay) so that only the sync differs
        run = fb
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    fb()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                fb()
            run = graph.replay
        except Exception:
            run = fb
        evs = []
        for i in range(args.warmup + min(args.steps, 20)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run()
            b.record()
            if i >= args.warmup:
                evs.append((a, b))
        torch.cuda.synchronize()
        fb_ms = sorted(a.elapsed_time(b) for a, b in evs)[len(evs) // 2]
    cb = cpu_baseline(name, desc, batch, world, fb_ms)
    step_ms = cb["sync_ms_per_iter"] + fb_ms
    out = {"impl": "reference", "metric": "images/sec", "value": cb["value"], "unit": "images/s", "n_gpus": world,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"{name} (batch {batch}/device, P={desc.param_count} fp32 params), synchronous SGD: "
                                  f"forward/backward + gradient sync + SGD update",
                      "global_batch": world * batch, "parallelism": f"dp{world}"},
           "impl_config": {"sync": "the reference's own socket_sync_cpu.cpp + parallel_cpu.cpp + socket.cpp (oracle/_ref, "
                                   f"{world} loopback processes on the host cores) + restated SGD update",
                           "producer": "the same PyTorch/cuDNN forward/backward as the GPU arm (CUDA-graph replay)",
                           "composition": "COMPOSED, not a joint loop: ms_per_step = median ms of the reference's "
                                          "sync+update loop (measured inside ref_sync, first iteration dropped) + "
                                          "median ms of forward/backward on the GPU; the two run back to back in "
                                          "the reference as well (solver.cpp:221-240), so they add"},
           "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "host_cores", "kind", "sample")},
           "split_ms": {"forward_backward": fb_ms, "reference_cpu_sync_and_update": cb["sync_ms_per_iter"]},
           "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    emit(out)


def run_reference_sweep(args):
    """Config 5, reference column: the reference's socket path (oracle/_ref) over the message sizes of the sweep
    at N = --gpus loopback ranks on THIS box's host cores (bounded: few iterations per point)."""
    rank, world = env_int("RANK", 0), env_int("WORLD_SIZE", 1)
    if rank != 0:
        return
    world = max(world, args.gpus, 2)
    from oracle import oracle as O
    if not O.ref_available():
        emit({"impl": "reference", "sweep": [], "unavailable": "oracle/_ref/ref_sync was not built"})
        return
    if args.sizes:
        sizes = [int(float(x) * (1 << 20)) // 4 * 4 for x in args.sizes.split(",")]
    else:
        sizes = [64 << 10, 256 << 10, 1 << 20, 4 << 20, 16 << 20, 64 << 20, 256 << 20]
    rows = []
    for S in sizes:
        P = S // 4
        iters = max(3, min(40, int(4000 / max(1.0, S / 1e6 * world))))
        r = O.run_ref_time(world, [P], iters=iters, lr_policy="fixed", base_lr=0.01, momentum=0.9, weight_decay=0.0005)
        rows.append({"bytes": S, "ranks": world, "iters": iters, "ms_per_iter": r["ms_per_iter_median"],
                     "ms_sync": r.get("ms_sync_median"), "cores": r.get("cores"),
                     "bus_gbs": S * 2 * (world - 1) / world / (r["ms_per_iter_median"] * 1e-3) / 1e9})
        print("[ref sweep] %8d KiB N=%d  %.3f ms/iter  bus %.3f GB/s" % (S >> 10, world, r["ms_per_iter_median"],
                                                                         rows[-1]["bus_gbs"]), file=sys.stderr)
    emit({"impl": "reference", "sweep": rows, "n_gpus": world, "host_cores": os.cpu_count(),
          "what": "reference socket_sync_cpu path (on_start + on_gradients_ready + restated update), loopback TCP"})


SWEEP_VARIANTS = {
    # name: (algo, options set BEFORE connect)
    "ldg": (1, {"kernel": 0, "nvls": 0}),
    "tma": (1, {"kernel": 1, "nvls": 0}),
    "push": (1, {"kernel": 2, "nvls": 0}),
    "push1": (1, {"kernel": 2, "nvls": 0, "push_vecs": 1}),
    "push4": (1, {"kernel": 2, "nvls": 0, "push_vecs": 4}),
    "push8": (1, {"kernel": 2, "nvls": 0, "push_vecs": 8}),
    "ll": (1, {"kernel": 4, "nvls": 0}),
    "ll1": (1, {"kernel": 4, "nvls": 0, "push_vecs": 1}),
    "ll4": (1, {"kernel": 4, "nvls": 0, "push_vecs": 4}),
    "ldg1s": (2, {"kernel": 0, "nvls": 0}),
    "tma1s": (2, {"kernel": 1, "nvls": 0}),
    "nvls1": (1, {"kernel": 3, "nvls": 1, "nvls_unroll": 1}),
    "nvls2": (1, {"kernel": 3, "nvls": 1, "nvls_unroll": 2}),
    "nvls4": (1, {"kernel": 3, "nvls": 1, "nvls_unroll": 4}),
    "nvls8": (1, {"kernel": 3, "nvls": 1, "nvls_unroll": 8}),
    "nvls1p": (1, {"kernel": 3, "nvls": 1, "nvls_unroll": 1, "nvls_p2p": 1}),
    "nvls2p": (1, {"kernel": 3, "nvls": 1, "nvls_unroll": 2, "nvls_p2p": 1}),
    "nvls3p": (1, {"kernel": 3, "nvls": 1, "nvls_unroll": 3, "nvls_p2p": 1}),
    "nvls4p": (1, {"kernel": 3, "nvls": 1, "nvls_unroll": 4, "nvls_p2p": 1}),
    "auto": (0, {}),
}
KERNEL_NAMES = {0: "ldg_stg_vector", 1: "tma_bulk_pipeline", 2: "push_store", 3: "nvls_multimem", 4: "ll_flagged_words"}


def run_sweep(args):
    """Config 5: all-reduce message sweep 64 KiB - 512 MiB (single segment), every kernel variant asked for
    with --variants, next to NCCL's all-reduce of the same message (which does not include the update)."""
    import torch
    import torch.distributed as dist
    import caffeonspark_b200 as C
    from caffeonspark_b200 import harness
    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    rows = []
    if args.sizes:
        sizes = [int(float(x) * (1 << 20)) // 4 * 4 for x in args.sizes.split(",")]
    else:
        sizes = [64 << 10, 256 << 10, 1 << 20, 4 << 20, 16 << 20, 64 << 20, 256 << 20, 512 << 20]
    sizes = [b for b in sizes if args.sweep_min_bytes <= b <= args.sweep_max_bytes]
    names = args.variants.split(",") if args.variants else (["ldg", "tma", "push", "auto"] if world > 1 else ["ldg", "tma"])
    if args.nvls == 1 and "nvls4" not in names:
        names.append("nvls4")
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for S in sizes:
        P = S // 4
        nccl_ms = None
        for vname in names:
            algo, opts = SWEEP_VARIANTS[vname]
            if world == 1 and (vname.startswith(("push", "nvls", "ll")) or algo == 2):
                continue
            desc = C.SolverDesc([P], lr_policy="fixed", base_lr=0.01, momentum=0.9, weight_decay=0.0005,
                                grad_dtype=args.grad_dtype)
            cl = harness.Cluster(desc, rank=rank, world=world, device=local)
            net = cl.net
            for k, v in opts.items():
                net.set_option(k, v)
            if world > 1 and algo:
                net.set_option("algo", algo)
            net.set_option("zero_diff", int(args.zero_diff))
            net.set_option("timing", 1)
            net.set_option("barrier_timeout_ms", 60000)
            cl.start()
            net.diff().normal_(0, 0.01)
            ms = []
            for i in range(args.warmup + args.steps):
                if S < (64 << 20):
                    flush_buf.zero_()
                torch.cuda.synchronize()
                if world > 1:
                    dist.barrier()
                net.sync_step(0)
                if not net.synchronize():
                    raise RuntimeError(net.last_error())
                if i >= args.warmup:
                    ms.append(net.last_kernel_ms())
            k = sorted(ms)[len(ms) // 2]
            if world > 1:
                t = torch.tensor([k], device="cuda", dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                k = float(t.item())
            # steady state: launches queued back to back on every rank (no host sync in between), so the
            # host-side launch skew between ranks is not part of the number
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 20
            net.set_option("timing", 0)
            st = torch.cuda.Stream()  # explicit stream: handle 0 would mean "the net's own stream"
            with torch.cuda.stream(st):
                if not net.sync_step(0, st.cuda_stream):
                    raise RuntimeError(net.last_error())
                a.record()
                for _ in range(reps):
                    if not net.sync_step(0, st.cuda_stream):
                        raise RuntimeError(net.last_error())
                b.record()
            torch.cuda.synchronize()
            if not net.synchronize():
                raise RuntimeError(net.last_error())
            piped = a.elapsed_time(b) / reps
            if world > 1:
                t = torch.tensor([piped], device="cuda", dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                piped = float(t.item())
            row = {"bytes": S, "variant": vname,
                   "algo": {0: "local", 1: "two_shot", 2: "one_shot"}[int(net.get_option("resolved_algo"))],
                   "kernel": KERNEL_NAMES[int(net.get_option("resolved_kernel"))],
                   "nvls_active": bool(net.get_option("nvls_active")), "grad_dtype": args.grad_dtype,
                   "zero_diff": bool(args.zero_diff),
                   "kernel_ms": k, "min_ms": min(ms), "pipelined_ms": piped}
            if args.trace and int(net.get_option("resolved_kernel")) != 1:
                # where the time goes inside one launch (CTA 0, %globaltimer); stamps per kernel:
                #  ldg/nvls: start, after barrier A, after reduce+update+push, after barrier B, after zero
                #  push    : start, after scatter-push, after barrier A, after reduce+update+push, after barrier B
                net.set_option("trace", 1)
                tr = []
                for _ in range(7):
                    torch.cuda.synchronize()
                    if world > 1:
                        dist.barrier()
                    net.sync_step(0)
                    net.synchronize()
                    t = [net.get_option(f"trace_{i}") for i in range(13)]
                    # phases, then inside barrier A and B: release fence, flag flight + peer lateness, acquire fence
                    tr.append([(t[i + 1] - t[i]) / 1e3 for i in range(4)] +
                              [(t[6] - t[5]) / 1e3, (t[7] - t[6]) / 1e3, (t[8] - t[7]) / 1e3,
                               (t[10] - t[9]) / 1e3, (t[11] - t[10]) / 1e3, (t[12] - t[11]) / 1e3])
                net.set_option("trace", 0)
                med = [round(sorted(c)[len(c) // 2], 2) for c in zip(*tr)]
                row["trace_us"] = med[:4]
                row["barrier_us_fence_wait_acquire"] = {"A": med[4:7], "B": med[7:10]}
            if world > 1:
                row["bus_gbs"] = S * 2 * (world - 1) / world / (k * 1e-3) / 1e9
            if world > 1 and nccl_ms is None:
                # NCCL all-reduce of the same message (the library baseline the fused kernel must beat);
                # it does NOT include the SGD update
                buf = torch.zeros(P, device="cuda")
                evs = []
                for i in range(args.warmup + args.steps):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    dist.barrier()
                    a.record()
                    dist.all_reduce(buf)
                    b.record()
                    torch.cuda.synchronize()
                    if i >= args.warmup:
                        evs.append(a.elapsed_time(b))
                nccl_ms = sorted(evs)[len(evs) // 2]
                t = torch.tensor([nccl_ms], device="cuda", dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                nccl_ms = float(t.item())
                del buf
            if world > 1:
                row["nccl_allreduce_ms"] = nccl_ms
            else:
                row["hbm_gbs"] = (24 if args.zero_diff else 20) * P / (k * 1e-3) / 1e9
            rows.append(row)
            if rank == 0:
                print("[sweep] %8d KiB %-7s %-18s nvls=%d  %.1f us (min %.1f, piped %.1f)  nccl %s  trace %s" % (
                    S >> 10, vname, row["kernel"], row["nvls_active"], k * 1e3, min(ms) * 1e3, piped * 1e3,
                    "%.1f us" % (nccl_ms * 1e3) if nccl_ms else "-",
                    (row.get("trace_us"), row.get("barrier_us_fence_wait_acquire"))), file=sys.stderr)
            net.deallocate()
            if world > 1:
                dist.barrier()
    if rank == 0:
        emit({"sweep": rows, "n_gpus": world, "unit": "ms / GB/s", "steps": args.steps})
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="caffenet", choices=["lenet", "cifar10_quick", "caffenet"],
                    help="default: CaffeNet batch 256/device (BASELINE config 4, the largest single-GPU config)")
    ap.add_argument("--extras", action="store_true", default=True,
                    help="also measure LeNet (config 2) and CIFAR-10-quick with the bf16 wire (config 3) as extra keys")
    ap.add_argument("--no-extras", dest="extras", action="store_false")
    ap.add_argument("--no-parity", action="store_true", help="N > 1: skip the seeded parity steps vs the oracle")
    ap.add_argument("--grad-dtype", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--algo", type=int, default=0, help="0 auto, 1 two-shot, 2 one-shot")
    ap.add_argument("--kernel", type=int, default=-1, help="-1 auto, 0 LDG/STG vector kernel, 1 TMA bulk-copy pipeline")
    ap.add_argument("--nvls", type=int, default=-1, help="NVSwitch multicast reduce/broadcast: -1 auto, 0 off, 1 on")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--kernels", action="store_true", default=True)
    ap.add_argument("--no-kernels", dest="kernels", action="store_false")
    ap.add_argument("--sweep", action="store_true")
    ap.add_argument("--trace", action="store_true", help="sweep: per-phase timestamps of the LDG kernel")
    ap.add_argument("--variants", default="", help="sweep: comma list of " + ",".join(SWEEP_VARIANTS))
    ap.add_argument("--sizes", default="", help="sweep: comma list of message sizes in MiB (fractions allowed)")
    ap.add_argument("--zero-diff", type=int, default=1, help="sweep: fold ClearParamDiffs into the kernel")
    ap.add_argument("--sweep-min-bytes", type=int, default=0)
    ap.add_argument("--sweep-max-bytes", type=int, default=1 << 40)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the weights, momentum history and loss that the last timed step of each workload "
                         "computed as DIR/<workload>_<name>.npy (float32; arrays over 4 Mi elements as a fixed sample)")
    args = ap.parse_args()
    args.warmup = max(3, args.warmup)
    if args.impl == "reference" and args.sweep:
        run_reference_sweep(args)
    elif args.impl == "reference":
        run_reference(args)
    elif args.sweep:
        run_sweep(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
