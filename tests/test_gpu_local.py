"""-m gpu parity: the fused SGD update at cluster_size == 1 (LocalCaffeNet) vs
the oracle, through the C ABI.  Bar: BIT-EXACT (the kernel uses explicitly
rounded, un-fused fp32 ops in the reference's order); the north-star tolerance
(1e-5 relative) is asserted as well so a failure reads in those terms."""
import numpy as np
import pytest

from gpu_util import Ranks, assert_bits_equal

pytestmark = pytest.mark.gpu

HP_LENET = dict(lr_policy="inv", base_lr=0.01, gamma=0.0001, power=0.75, momentum=0.9, weight_decay=0.0005)
HP_CIFAR = dict(lr_policy="fixed", base_lr=0.001, momentum=0.9, weight_decay=0.004)

LAYOUTS = {
    "lenet": ([500, 20, 25000, 50, 400000, 500, 5000, 10], [1, 2] * 4, [1, 1] * 4, HP_LENET),
    "cifar10_quick": ([2400, 32, 25600, 32, 51200, 64, 65536, 64, 640, 10], [1, 2] * 5, [1, 1] * 5, HP_CIFAR),
    "ragged_tiny_blobs": ([3, 1, 2, 5, 1, 1, 7, 1021, 2, 1], [1, 2, 1, 2, 1, 2, 1, 2, 1, 2],
                          [1, 0, 1, 0, 1, 0, 1, 1, 0, 1], HP_LENET),
    "single_element": ([1], [1], [1], HP_CIFAR),
    "not_multiple_of_4": ([4099], [1], [1], dict(lr_policy="step", base_lr=0.01, gamma=0.1, stepsize=2,
                                                 momentum=0.9, weight_decay=0.0005)),
}


@pytest.mark.parametrize("name", sorted(LAYOUTS))
@pytest.mark.parametrize("bf16", [False, True])
@pytest.mark.parametrize("kernel", [0, 1], ids=["ldg", "tma"])
def test_local_update_bit_exact(cos, oracle, name, bf16, kernel):
    counts, lm, dm, hp = LAYOUTS[name]
    desc = cos.SolverDesc(counts, lm, dm, grad_dtype="bf16" if bf16 else "fp32", **hp)
    sim = oracle.Simulation(1, counts, lm, dm, seed=7, bf16=bf16, **hp)
    R = Ranks(cos, desc, 1, kernel=kernel)
    try:
        R.set_weights([sim.data[0]])
        R.connect()
        for t in range(5):
            g = oracle.fill(sim.P, 7, (t + 1) * 4096, 0.01)  # raw fp32 gradient; bf16 rounding happens in-kernel
            rate = sim.step([sim.gradient(0, t)])
            assert np.float32(R.nets[0].learning_rate()).tobytes() == np.float32(rate).tobytes()
            R.step([g])
            assert R.nets[0].iter() == sim.iter
            w, h = R.weights(0), R.history(0)
            assert np.allclose(w, sim.data[0], rtol=1e-5, atol=0)
            assert_bits_equal(w, sim.data[0], f"{name} weights iter {t}")
            assert_bits_equal(h, sim.hist[0], f"{name} history iter {t}")
            assert not R.diff(0).any(), "ClearParamDiffs fold: diff_ must be zero after the step"
    finally:
        R.close()


def test_zero_diff_can_be_disabled(cos, oracle):
    counts = [1000, 24]
    desc = cos.SolverDesc(counts, **HP_CIFAR)
    R = Ranks(cos, desc, 1, zero_diff=0)
    try:
        R.connect()
        g = oracle.fill(1024, 3, 1, 0.01)
        R.step([g])
        assert_bits_equal(R.diff(0), g, "diff_ untouched when zero_diff=0")
    finally:
        R.close()


def test_boundary_conventions_like_CaffeNetTest(cos, tmp_path):
    # CaffeNetTest.java:86-159 on a local net
    prefix = str(tmp_path / "cos_test_local")
    desc = cos.SolverDesc([100, 10], max_iter=2000, snapshot_prefix=prefix, **HP_CIFAR)
    net = cos.CaffeNet(desc)
    try:
        assert net.init(-1) is False
        assert net.deviceID(-1) == -1
        assert net.getInitIter(-1) == -1
        assert net.getMaxIter(-1) == -1
        assert net.snapshotFilename(-1, False) is None
        assert net.connect(None) is True                      # connectnull
        addrs = net.localAddresses()
        assert len(addrs) == 0                                # testBasic
        assert net.connect(addrs)
        assert net.sync() is True
        assert net.deviceID(0) == 0
        assert net.init(0, True)
        assert net.getInitIter(0) == 0
        assert net.getMaxIter(0) == 2000
        it = net.snapshot()
        assert it >= 0
        import os
        for is_state in (True, False):
            fn = net.snapshotFilename(it, is_state)
            assert fn.startswith(prefix + "_iter_0") and os.path.exists(fn)
            os.unlink(fn)
        with pytest.raises(cos.CosError, match="data is NULL"):  # trainnull
            net.train(0, None)
        assert net.train(0, [np.zeros((2, 1, 2, 2), np.float32), np.zeros((2,), np.float32)]) is False
        assert "gradient producer" in net.last_error()
    finally:
        net.deallocate()


def test_socket_net_connectbogus(cos):
    # CaffeNetTest.java:116-126: SocketCaffeNet.connect({"0x222","0x333"}) must fail, not hang
    desc = cos.SolverDesc([64], **HP_CIFAR)
    net = cos.CaffeNet(desc, "", "", 1, 2, 0, False, cos.CaffeNet.SOCKET, -1, 0)
    try:
        la = net.localAddresses()
        assert len(la) == 2 and la[0] == "" and la[1].startswith("cosb200://")
        assert net.connect(["0x222", "0x333"]) is False
        assert net.sync_step(0) is False and "connect" in net.last_error()
    finally:
        net.deallocate()
    with pytest.raises(cos.CosError, match="unable to create CaffeNet"):
        cos.CaffeNet(desc, "", "", 1, 2, 0, False, cos.CaffeNet.NONE, -1, 0)


@pytest.mark.parametrize("kernel", [0, 1], ids=["ldg", "tma"])
def test_full_size_caffenet_properties(cos, oracle, kernel):
    """BASELINE full size (P = 60,965,224): oracle comparison on the whole
    buffer (the C oracle handles it in seconds) + a size-independent property:
    with zero gradient, zero decay multipliers and zero history the weights
    must not move (idempotence)."""
    from caffeonspark_b200 import nets
    desc = nets.solver_desc("caffenet")
    assert desc.param_count == 60965224
    sim = oracle.Simulation(1, desc.counts, desc.lr_mult, desc.decay_mult, seed=5, **desc.hyper())
    R = Ranks(cos, desc, 1, kernel=kernel, timing=1)
    try:
        R.set_weights([sim.data[0]])
        R.connect()
        for t in range(2):
            g = sim.gradient(0, t)
            sim.step([g])
            R.step([g])
        assert_bits_equal(R.weights(0), sim.data[0], "caffenet weights")
        assert_bits_equal(R.history(0), sim.hist[0], "caffenet history")
        ms = R.nets[0].last_kernel_ms()
        assert 0 < ms < 1.0, ms  # 24P = 1.46 GB in ~0.23 ms on a B200 (0.95+ of the HBM copy peak); loose 4x guard
    finally:
        R.close()
    desc0 = cos.SolverDesc([60965224], [1.0], [0.0], lr_policy="fixed", base_lr=0.1, momentum=0.9, weight_decay=0.5)
    R = Ranks(cos, desc0, 1, kernel=kernel)
    try:
        w0 = oracle.fill(desc0.param_count, 9, 0, 0.05)
        R.set_weights([w0])
        R.connect()
        R.step([np.zeros_like(w0)])
        assert_bits_equal(R.weights(0), w0, "idempotence under zero gradient")
    finally:
        R.close()


def test_snapshot_restore_resumes_bit_exactly(cos, oracle, tmp_path):
    """Checkpoint/resume (CaffeNet.cpp:196-205 restore path, CaffeProcessor.scala:454-465 snapshot):
    snapshot at iteration 2, resume in a NEW net from the files, and the continued run must equal the
    uninterrupted one bit for bit (weights, history, iteration counter, learning-rate schedule)."""
    from caffeonspark_b200 import nets
    from gpu_util import to_dev, to_host
    import torch
    (tmp_path / "net.prototxt").write_text(nets.net_prototxt("cifar10_quick"))
    prefix = str(tmp_path / "ckpt")
    (tmp_path / "solver.prototxt").write_text(
        f'net: "net.prototxt"\nbase_lr: 0.01\nmomentum: 0.9\nweight_decay: 0.004\nlr_policy: "inv"\n'
        f'gamma: 0.01\npower: 0.75\nmax_iter: 100\nsnapshot_prefix: "{prefix}"\n')
    solver = str(tmp_path / "solver.prototxt")
    P = nets.EXPECTED_PARAM_COUNT["cifar10_quick"]
    grads = [oracle.fill(P, 21, 4096 * (t + 1), 0.01) for t in range(4)]

    def run_steps(net, ts):
        for t in ts:
            to_dev(net.diff(), grads[t])
            torch.cuda.synchronize()
            assert net.sync_step(0) and net.synchronize(), net.last_error()

    a = cos.CaffeNet(solver)
    try:
        assert a.connect(a.localAddresses())
        to_dev(a.data(), oracle.fill(P, 21, 0, 0.05))
        run_steps(a, [0, 1])
        it = a.snapshot()
        assert it == 2
        model, state = a.snapshotFilename(it, False), a.snapshotFilename(it, True)
        rate_at_2 = a.learning_rate()
        w_at_2 = to_host(a.data())
        run_steps(a, [2, 3])
        w_ref, h_ref = to_host(a.data()), to_host(a.history())
    finally:
        a.deallocate()
    b = cos.CaffeNet(solver, model, state)
    try:
        assert b.connect(b.localAddresses())
        assert b.getInitIter(0) == 2 and b.iter() == 2
        assert np.float32(b.learning_rate()).tobytes() == np.float32(rate_at_2).tobytes()
        run_steps(b, [2, 3])
        assert b.iter() == 4
        assert_bits_equal(to_host(b.data()), w_ref, "weights after resume")
        assert_bits_equal(to_host(b.history()), h_ref, "history after resume")
    finally:
        b.deallocate()
    assert model.endswith("ckpt_iter_2.caffemodel") and state.endswith("ckpt_iter_2.solverstate")
    # layer-wise content, readable by stock Caffe: conv1 weights are [32, 3, 5, 5]
    assert cos.read_caffemodel_blob(model, "conv1", 0).size == 2400
    assert cos.read_solverstate(state)[0] == 2
    with pytest.raises(cos.CosError, match="not a SolverState"):
        cos.CaffeNet(solver, state, model)  # swapped files must be rejected
    c = cos.CaffeNet(solver, model, "")     # weights only (copyLayers), iteration restarts at 0
    try:
        assert c.getInitIter(0) == 0
        assert_bits_equal(to_host(c.data()), w_at_2, "copyLayers restores the weights")
    finally:
        c.deallocate()


def test_hdf5_snapshot_and_resume(cos, oracle, tmp_path):
    """The reference's own cifar10_quick_solver.prototxt asks for snapshot_format: HDF5 (solver.cpp:417-418,
    sgd_solver.cpp:251-252,279-301, net.cpp:867-917).  snapshot() then writes <prefix>_iter_<n>.caffemodel.h5 /
    .solverstate.h5 (the names CaffeNet.java:203-205 computes) as real HDF5 (csrc/hdf5_io.cpp), and a new net
    resumed from them continues bit-exactly (RestoreSolverStateFromHDF5 / CopyTrainedLayersFromHDF5)."""
    from caffeonspark_b200 import nets
    from gpu_util import to_dev, to_host
    import torch
    (tmp_path / "net.prototxt").write_text(nets.net_prototxt("cifar10_quick"))
    (tmp_path / "solver.prototxt").write_text(
        f'net: "net.prototxt"\nbase_lr: 0.001\nmomentum: 0.9\nweight_decay: 0.004\nlr_policy: "step"\ngamma: 0.5\n'
        f'stepsize: 2\nmax_iter: 10\nsnapshot_format: HDF5\nsnapshot_prefix: "{tmp_path / "c10"}"\n')
    solver = str(tmp_path / "solver.prototxt")
    P = nets.EXPECTED_PARAM_COUNT["cifar10_quick"]
    grads = [oracle.fill(P, 23, 4096 * (t + 1), 0.01) for t in range(4)]

    def run_steps(net, ts):
        for t in ts:
            to_dev(net.diff(), grads[t])
            torch.cuda.synchronize()
            assert net.sync_step(0) and net.synchronize(), net.last_error()

    a = cos.CaffeNet(solver)
    try:
        assert a.connect(a.localAddresses())
        to_dev(a.data(), oracle.fill(P, 23, 0, 0.05))
        run_steps(a, [0, 1, 2])
        assert a.snapshot() == 3, a.last_error()
        model, state = a.snapshotFilename(3, False), a.snapshotFilename(3, True)
        assert model.endswith("c10_iter_3.caffemodel.h5") and state.endswith("c10_iter_3.solverstate.h5")
        assert open(model, "rb").read(8) == b"\x89HDF\r\n\x1a\n" and open(state, "rb").read(8) == b"\x89HDF\r\n\x1a\n"
        w3 = to_host(a.data())
        run_steps(a, [3])
        w_ref, h_ref = to_host(a.data()), to_host(a.history())
    finally:
        a.deallocate()
    assert cos.read_caffemodel_blob(model, "conv1", 0).size == 2400        # /data/conv1/0
    it, step, learned, hist = cos.read_solverstate(state)
    assert (it, step, learned) == (3, 1, model) and len(hist) == 10
    b = cos.CaffeNet(solver, "", state)  # Solver::Restore follows learned_net for the weights
    try:
        assert b.connect(b.localAddresses())
        assert b.iter() == 3
        assert_bits_equal(to_host(b.data()), w3, "weights restored from the .caffemodel.h5")
        run_steps(b, [3])
        assert_bits_equal(to_host(b.data()), w_ref, "weights after resuming from HDF5")
        assert_bits_equal(to_host(b.history()), h_ref, "history after resuming from HDF5")
    finally:
        b.deallocate()


def test_device_fill_is_the_oracles_generator(cos, oracle):
    """cos_net_fill (used by bench.py's N > 1 parity steps so that no 4P-byte tensor crosses PCIe) must produce
    exactly the oracle driver's seeded tensors."""
    desc = cos.SolverDesc([100003, 5], **HP_CIFAR)
    net = cos.CaffeNet(desc)
    try:
        assert net.connect(net.localAddresses())
        for which, view, seed, stream, amp in (("data", net.data, 42, 0, 0.05), ("diff", net.diff, 1234, 3 * 4096 + 7, 0.01),
                                               ("history", net.history, 2**40 + 1, 2**33, 1.0)):
            net.fill(which, seed, stream, amp)
            assert_bits_equal(view().cpu().numpy(), oracle.fill(100008, seed, stream, amp), f"device fill of {which}")
        with pytest.raises(cos.CosError):
            net.fill(7, 1, 1, 1.0)
    finally:
        net.deallocate()


@pytest.mark.parametrize("kernel", [0, 1], ids=["ldg", "tma"])
def test_l1_regularization_bit_exact(cos, oracle, kernel):
    """regularization_type: "L1" (sgd_solver.cpp:161-168) on the fused update path, incl. sign(+-0) = 0."""
    counts, lm, dm = [1021, 7, 64], [1, 2, 1], [1, 0, 0.5]
    hp = dict(lr_policy="fixed", base_lr=0.01, momentum=0.9, weight_decay=0.004)
    desc = cos.SolverDesc(counts, lm, dm, regularization_type="L1", **hp)
    sim = oracle.Simulation(1, counts, lm, dm, seed=17, regularization_type="L1", **hp)
    sim.data[0][:4] = [0.0, -0.0, 0.5, -0.5]
    R = Ranks(cos, desc, 1, kernel=kernel)
    try:
        R.set_weights([sim.data[0]])
        R.connect()
        for t in range(3):
            g = sim.gradient(0, t)
            sim.step([g])
            R.step([g])
            assert_bits_equal(R.weights(0), sim.data[0], f"L1 weights iter {t}")
            assert_bits_equal(R.history(0), sim.hist[0], f"L1 history iter {t}")
    finally:
        R.close()
