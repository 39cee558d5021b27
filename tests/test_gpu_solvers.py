"""-m gpu parity of the Nesterov, AdaGrad, RMSProp and AdaDelta solvers on the fused sync kernels (LDG, push,
LL): weights, history and AdaDelta's second history bit-exact against the solver oracle (tests/solver_oracle.py),
diff_ zero after every step; the kernel routing of a non-SGD solver; AdaDelta snapshot / restore; train()."""
import os
import re
import socket
import sys

import numpy as np
import pytest

import solver_oracle as SO
from conftest import ROOT, gpu_count
from gpu_util import Ranks, assert_bits_equal, to_host

pytestmark = pytest.mark.gpu

TYPES = ("Nesterov", "AdaGrad", "RMSProp", "AdaDelta")
BASE = dict(lr_policy="inv", base_lr=0.01, gamma=0.0001, power=0.75, weight_decay=0.0005)
SOLVER_HP = {  # hyper-parameters of the reference's example solvers
    "SGD": dict(momentum=0.9),
    "Nesterov": dict(momentum=0.95),
    "AdaGrad": dict(momentum=0.0, delta=1e-8),
    "RMSProp": dict(momentum=0.0, rms_decay=0.98, delta=1e-8),
    "AdaDelta": dict(momentum=0.95, delta=1e-6),
}
LAYOUTS = {  # the layouts of test_gpu_local.py that exercise the scalar head / tail and blob boundaries
    "ragged_tiny_blobs": ([3, 1, 2, 5, 1, 1, 7, 1021, 2, 1], [1, 2, 1, 2, 1, 2, 1, 2, 1, 2],
                          [1, 0, 1, 0, 1, 0, 1, 1, 0, 1]),
    "single_element": ([1], [1], [1]),
    "not_multiple_of_4": ([4099], [1], [1]),
}


def _hp(type, **kw):
    return dict(BASE, type=type, **SOLVER_HP[type], **kw)


def _check(R, sim, N, what):
    cw, ch, ch2 = sim.consistent_weights(), sim.consistent_history(), sim.consistent_history2()
    mode = R.nets[0].get_option("resolved_algo")
    for r in range(N):
        net = R.nets[r]
        assert_bits_equal(R.weights(r), cw, f"{what} weights rank {r}")
        o, s = (0, sim.P) if mode in (0, 2) else net.shard()  # two-shot: the history is valid on the owner only
        assert_bits_equal(R.history(r)[o:o + s], ch[o:o + s], f"{what} history rank {r}")
        if ch2 is None:
            assert net.update_history() is None
        else:
            assert_bits_equal(to_host(net.update_history())[o:o + s], ch2[o:o + s], f"{what} h2 rank {r}")
        assert not R.diff(r).any(), f"{what}: diff_ must be zero after the step"


def _run(cos, N, counts, lm, dm, type, iters=4, seed=11, bf16=False, expect_kernel=None, **opts):
    hp = _hp(type, regularization_type="L2")
    desc = cos.SolverDesc(counts, lm, dm, grad_dtype="bf16" if bf16 else "fp32", **hp)
    sim = SO.Simulation(N, counts, lm, dm, seed=seed, bf16=bf16, **hp)
    R = Ranks(cos, desc, N, **opts)
    try:
        if expect_kernel is not None:
            assert R.nets[0].get_option("resolved_kernel") == expect_kernel
        R.set_weights(sim.data)
        R.connect()
        for t in range(iters):
            grads = [SO.O.fill(sim.P, seed, (t + 1) * 4096 + r, 0.01) for r in range(N)]  # bf16 rounding in-kernel
            sim.step()
            R.step(grads)
            _check(R, sim, N, f"{type} N={N} iter {t}")
    finally:
        R.close()


@pytest.mark.parametrize("type", TYPES)
@pytest.mark.parametrize("name", sorted(LAYOUTS))
@pytest.mark.parametrize("bf16", [False, True])
def test_local_ldg_bit_exact(cos, type, name, bf16):
    _run(cos, 1, *LAYOUTS[name], type, iters=5, bf16=bf16, expect_kernel=0)


@pytest.mark.parametrize("type", TYPES)
@pytest.mark.parametrize("N", [2, 3, 4])
@pytest.mark.parametrize("kernel,algo", [(2, 1), (4, 1), (0, 1), (0, 2)], ids=["push", "ll", "ldg2shot", "ldg1shot"])
def test_in_process_bit_exact(cos, type, N, kernel, algo):
    counts, lm, dm = [5000, 20, 2500, 50, 7, 1], [1, 2, 1, 2, 1, 2], [1, 0, 1, 1, 0, 1]
    _run(cos, N, counts, lm, dm, type, iters=3, kernel=kernel, algo=algo, expect_kernel=kernel,
         bf16=(kernel == 2 and N == 3))


@pytest.mark.parametrize("type", ["AdaGrad", "AdaDelta"])
def test_forced_variants_fall_back(cos, type):
    """TMA and NVLS run SGD only: a forced kernel 1 runs LDG, a forced kernel 3 AUTO's choice, and one-shot at
    2 MiB or more uses LDG where SGD uses TMA."""
    counts, lm, dm = [3000, 17], [1, 2], [1, 0]
    _run(cos, 1, counts, lm, dm, type, iters=2, kernel=1, expect_kernel=0)
    auto = Ranks(cos, cos.SolverDesc(counts, lm, dm, **_hp(type)), 2, algo=1)
    want = auto.nets[0].get_option("resolved_kernel")
    auto.close()
    assert want == 4  # LL for this size
    _run(cos, 2, counts, lm, dm, type, iters=2, kernel=3, algo=1, expect_kernel=want)
    _run(cos, 2, counts, lm, dm, type, iters=2, kernel=1, algo=1, expect_kernel=0)
    big = [600000, 3]  # 2.4 MB
    sgd = Ranks(cos, cos.SolverDesc(big, [1, 1], [1, 1], **_hp("SGD")), 2, algo=2)
    assert sgd.nets[0].get_option("resolved_kernel") == 1
    sgd.close()
    _run(cos, 2, big, [1, 1], [1, 1], type, iters=2, algo=2, expect_kernel=0)


NET = ('name: "solvers" layer { name: "data" type: "Input" top: "x" input_param { shape { dim: 4 dim: 77 } } }\n'
       'layer { name: "ip1" type: "InnerProduct" bottom: "x" top: "y" inner_product_param { num_output: 33 } }\n'
       'layer { name: "ip2" type: "InnerProduct" bottom: "y" top: "z" inner_product_param { num_output: 5 } }\n')


def _prototxt_ranks(cos, solver, N, model="", state=""):
    R = Ranks.__new__(Ranks)
    R.cos, R.N, R.nets = cos, N, []
    for r in range(N):
        net = cos.CaffeNet(solver, model, state, 1, N, r, True, cos.CaffeNet.SOCKET, -1, 0)
        for k, v in dict(barrier_timeout_ms=8000, grid=4, block=128, initial_gather=0, algo=1).items():
            net.set_option(k, v)
        R.nets.append(net)
    return R


@pytest.mark.parametrize("fmt", ["BINARYPROTO", "HDF5"])
def test_adadelta_snapshot_restore_continue(cos, tmp_path, fmt):
    N, seed = 2, 23
    (tmp_path / "net.prototxt").write_text(NET)
    solver = tmp_path / "solver.prototxt"
    solver.write_text(f'net: "net.prototxt"\ntype: "AdaDelta"\nbase_lr: 1.0\nmomentum: 0.95\ndelta: 1e-6\n'
                      f'weight_decay: 0.0005\nlr_policy: "fixed"\nsnapshot_prefix: "{tmp_path}/snap"\n'
                      f'snapshot_format: {fmt}\n')
    desc = cos.parse_solver(str(solver))
    counts = desc.counts
    sim = SO.Simulation(N, counts, desc.lr_mult, desc.decay_mult, seed=seed, lr_policy="fixed", base_lr=1.0,
                        momentum=desc.momentum, weight_decay=desc.weight_decay, type="AdaDelta", delta=desc.delta)
    grads = [[SO.O.fill(sim.P, seed, (t + 1) * 4096 + r, 0.01) for r in range(N)] for t in range(5)]
    R = _prototxt_ranks(cos, str(solver), N)
    try:
        R.set_weights(sim.data)
        R.connect()
        for t in range(5):
            sim.step()
            R.step(grads[t])
            _check(R, sim, N, f"uninterrupted iter {t}")
            if t == 1:
                it = R.nets[0].snapshot()
                assert it == 2
                state, model = R.nets[0].snapshotFilename(it, True), R.nets[0].snapshotFilename(it, False)
                s_iter, _, _, hist = cos.read_solverstate(state)
                assert s_iter == 2 and [h.size for h in hist] == counts + counts  # h of every blob, then h2
                assert_bits_equal(np.concatenate(hist[:len(counts)]), sim.consistent_history(), "snapshot h")
                assert_bits_equal(np.concatenate(hist[len(counts):]), sim.consistent_history2(), "snapshot h2")
        final = R.weights(0)
    finally:
        R.close()
    R = _prototxt_ranks(cos, str(solver), N, model, state)
    try:
        R.connect()
        assert R.nets[0].iter() == 2
        for t in range(2, 5):
            R.step(grads[t])
        for r in range(N):
            assert_bits_equal(R.weights(r), final, f"restored run rank {r}")
            assert not R.diff(r).any()
    finally:
        R.close()
    bad = tmp_path / "sgd.prototxt"  # a one-history snapshot does not fit AdaDelta, and the other way round
    bad.write_text(solver.read_text().replace('type: "AdaDelta"', 'type: "SGD"'))
    with pytest.raises(cos.CosError, match="history blobs"):
        cos.CaffeNet(str(bad), model, state, 1, 1, 0, True, cos.CaffeNet.NONE, -1, 0)


@pytest.mark.parametrize("type", TYPES)
def test_train_lenet_from_prototxt(cos, tmp_path, type):
    import torch
    from caffeonspark_b200 import harness, nets
    solver = nets.write_prototxts("lenet", str(tmp_path))
    text = re.sub(r"momentum: \S+\n", f"momentum: {SOLVER_HP[type]['momentum']}\n", open(solver).read())
    extra = "".join(f"{k}: {v}\n" for k, v in SOLVER_HP[type].items() if k != "momentum")
    open(solver, "w").write(text + f'type: "{type}"\n' + extra)
    net = cos.CaffeNet(solver, "", "", 1, 1, 0, True, cos.CaffeNet.NONE, -1, 0)
    try:
        assert net.connect(net.localAddresses()) and net.init(0, True)
        net.set_option("zero_diff", 0)  # keep the gradient so the test can feed it to the oracle
        prod = harness.make_producer("lenet", net)
        desc = net.desc
        assert desc.type == type
        rng = np.random.RandomState(0)
        x = torch.from_numpy(rng.rand(64, 1, 28, 28).astype(np.float32)).pin_memory()
        y = torch.from_numpy(rng.randint(0, 10, (64, 1, 1, 1)).astype(np.float32)).pin_memory()
        for t in range(6):
            w, h = to_host(net.data()), to_host(net.history())
            h2 = to_host(net.update_history()) if type == "AdaDelta" else None
            net.diff().zero_()
            torch.cuda.synchronize()
            rate = net.learning_rate()
            assert net.train(0, [x, y]), net.last_error()
            assert net.synchronize(), net.last_error()
            g = to_host(net.diff())  # the gradient the producer accumulated
            SO.apply_update(0, desc.param_count, w, g.copy(), h, h2, desc.counts, desc.lr_mult, desc.decay_mult,
                            np.float32(rate), np.float32(desc.momentum), np.float32(desc.weight_decay), type=type,
                            delta=desc.delta, rms_decay=desc.rms_decay)
            assert_bits_equal(to_host(net.data()), w, f"{type} weights after train() iter {t}")
            assert_bits_equal(to_host(net.history()), h, f"{type} history after train() iter {t}")
            if h2 is not None:
                assert_bits_equal(to_host(net.update_history()), h2, f"{type} h2 after train() iter {t}")
        assert np.isfinite(net.last_loss()) and prod is not None
    finally:
        net.deallocate()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, type, counts, bf16, kernel, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch
    import torch.distributed as dist
    import caffeonspark_b200 as C
    import solver_oracle
    from caffeonspark_b200.harness import Cluster
    from gpu_util import to_dev
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{rank}"))
    try:
        lm, dm = [1, 2] * (len(counts) // 2), [1, 0] * (len(counts) // 2)
        hp = _hp(type)
        desc = C.SolverDesc(counts, lm, dm, grad_dtype="bf16" if bf16 else "fp32", **hp)
        sim = solver_oracle.Simulation(world, counts, lm, dm, seed=77, bf16=bf16, **hp)
        cl = Cluster(desc, rank=rank, world=world, device=rank)
        net = cl.net
        net.set_option("barrier_timeout_ms", 15000)
        if kernel is not None:
            net.set_option("kernel", kernel)
        to_dev(net.data(), sim.data[rank])
        torch.cuda.synchronize()
        cl.start()
        ok = True
        for t in range(2):
            g = solver_oracle.O.fill(sim.P, 77, (t + 1) * 4096 + rank, 0.01)
            sim.step()
            to_dev(net.diff(), g)
            torch.cuda.synchronize()
            assert net.sync_step(0), net.last_error()
            assert net.synchronize(), net.last_error()
            o, s = net.shard()
            ok = ok and np.array_equal(to_host(net.data()).view(np.uint32), sim.consistent_weights().view(np.uint32))
            ok = ok and np.array_equal(to_host(net.history())[o:o + s].view(np.uint32),
                                       sim.consistent_history()[o:o + s].view(np.uint32))
            if type == "AdaDelta":
                ok = ok and np.array_equal(to_host(net.update_history())[o:o + s].view(np.uint32),
                                           sim.consistent_history2()[o:o + s].view(np.uint32))
            ok = ok and not bool(net.diff().any())
        q.put((rank, bool(ok), int(net.get_option("resolved_kernel"))))
        assert net.sync()
        net.deallocate()
    finally:
        dist.destroy_process_group()


def _multiproc(world, type, counts, bf16=False, kernel=None):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, type, counts, bf16, kernel, q)) for r in range(world)]
    [p.start() for p in procs]
    [p.join(600) for p in procs]
    for p in procs:
        if p.is_alive():
            p.kill()
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    res = sorted(q.get(timeout=5) for _ in range(world))
    assert all(ok for _, ok, _ in res), res
    return {k for _, _, k in res}


SMALL = [500, 20, 25000, 50, 400000, 500, 5000, 10]  # LeNet layout


@pytest.mark.skipif(gpu_count() < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("type", TYPES)
@pytest.mark.parametrize("kernel", [None, 2, 0], ids=["auto", "push", "ldg"])
def test_one_process_per_gpu(cos, type, kernel):
    for world in sorted({2, min(gpu_count(), 8)}):
        _multiproc(world, type, SMALL, bf16=(type == "RMSProp"), kernel=kernel)


@pytest.mark.skipif(gpu_count() < 6, reason="needs >= 6 GPUs")
def test_adadelta_large_layout_runs_on_push_not_nvls(cos):
    """32 MiB or more at N >= 6 is where SGD runs on NVLS; AdaDelta resolves to push and stays bit-exact."""
    counts = [8_400_000, 1000, 7, 13]  # 33.6 MB
    assert _multiproc(min(gpu_count(), 8), "AdaDelta", counts) == {2}
