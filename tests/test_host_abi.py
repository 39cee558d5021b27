"""CPU tests of the product library's host side: the C ABI loads and exports
every symbol include/caffedistri_b200.h declares, the pure host functions
(chunk, learning rate, prototxt layout parser) agree with the oracle / the
reference's config files, and compute entry points FAIL LOUDLY without a GPU.
No device compute is attempted here."""
import ctypes
import json
import os
import re

import numpy as np
import pytest

from conftest import ROOT, gpu_count


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "caffedistri_b200.h")).read()
    return sorted(set(re.findall(r"COS_API[^;(]*?\b(cos_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(cos):
    from caffeonspark_b200 import _lib
    names = _header_symbols()
    assert len(names) >= 40
    L = ctypes.CDLL(cos.library_path())
    for n in names:
        assert hasattr(L, n), f"{n} declared in the header but not exported"
    bound = {s[0] for s in _lib.SYMBOLS}
    assert set(names) == bound, f"ctypes table out of sync with the header: {set(names) ^ bound}"
    assert b"sm_100a" in _lib.lib().cos_version()


def test_no_libcuda_link_dependency(cos):
    # the library must load on a GPU-less box: driver API only via cudaGetDriverEntryPoint
    import subprocess
    out = subprocess.run(["ldd", cos.library_path()], capture_output=True, text=True).stdout
    assert "libcuda.so" not in out and "libnccl" not in out


def test_chunk_matches_oracle_bit_exact(cos, oracle):
    rng = np.random.RandomState(5)
    cases = [(431080, 8), (145578, 4), (60965224, 8), (1, 2), (5, 8), (2 ** 33 + 7, 7)]
    cases += [(int(rng.randint(1, 10 ** 9)), int(rng.randint(1, 17))) for _ in range(200)]
    for P, N in cases:
        for r in range(N):
            assert cos.chunk(P, N, r) == oracle.chunk(P, N, r)


def test_learning_rate_matches_oracle_bit_exact(cos, oracle):
    pol = [("fixed", {}), ("inv", dict(gamma=1e-4, power=0.75)), ("step", dict(gamma=0.1, stepsize=7)),
           ("exp", dict(gamma=0.999)), ("poly", dict(power=1.5, max_iter=500)),
           ("sigmoid", dict(gamma=-0.01, stepsize=200)), ("multistep", dict(gamma=0.5, stepvalues=(3, 50, 400)))]
    for name, kw in pol:
        st = oracle.LrState()
        step = 0
        for it in list(range(0, 60)) + [399, 400, 401, 499]:
            want = oracle.learning_rate(name, 0.01, it=it, state=st, **kw)
            got, step = cos.learning_rate(name, 0.01, it=it, current_step=step, **kw)
            assert np.float32(got).tobytes() == np.float32(want).tobytes(), (name, it, got, want)
    with pytest.raises(cos.CosError):
        cos.learning_rate("bogus", 0.1)


def test_layout_parser_on_generated_prototxt(cos, tmp_path):
    from caffeonspark_b200 import nets
    for name, P in nets.EXPECTED_PARAM_COUNT.items():
        solver = nets.write_prototxts(name, str(tmp_path))
        d = cos.parse_solver(solver)
        counts, lm, dm, _ = nets.layout(name)
        assert d.counts == counts and d.lr_mult == lm and d.decay_mult == dm
        assert d.param_count == P
        s = nets.NETS[name]["solver"]
        assert d.lr_policy == s["lr_policy"] and d.max_iter == s["max_iter"]
        assert d.base_lr == pytest.approx(s["base_lr"]) and d.momentum == pytest.approx(s["momentum"])
        assert d.batch_size == nets.NETS[name]["batch"]


CONFIGS = os.path.join(ROOT, "tests", "golden", "configs")


def test_layout_parser_on_reference_config_files(cos):
    # SURVEY.md App. D: the reference's own prototxts (its data/ and caffe-distri/src/test/resources/ files,
    # stored under tests/golden/configs) must yield these layouts
    want = {"lenet_memory_solver.prototxt": (431080, 8, "inv", 64),
            "cifar10_quick_solver.prototxt": (145578, 10, "fixed", 100),
            "bvlc_reference_solver.prototxt": (60965224, 16, "step", 2),
            "lenet_cos_solver.prototxt": (431080, 8, None, None)}
    for f, (P, nblobs, pol, batch) in want.items():
        d = cos.parse_solver(os.path.join(CONFIGS, "data", f))
        assert d.param_count == P and len(d.counts) == nblobs
        if pol:
            assert d.lr_policy == pol and d.batch_size == batch
    d = cos.parse_solver(os.path.join(CONFIGS, "data", "bvlc_reference_solver.prototxt"))
    assert d.decay_mult[1::2] == [0.0] * 8 and d.lr_mult[1::2] == [2.0] * 8  # biases: lr 2, decay 0
    # every other CaffeOnSpark configuration on the path: DataFrame-fed LeNet and the JNI test's CaffeNet
    # (fc8 with 2 outputs: 60,965,224 - (4,096,000 + 1000) + (4096 * 2 + 2))
    assert cos.parse_solver(os.path.join(CONFIGS, "data", "lenet_dataframe_solver.prototxt")).param_count == 431080
    t = cos.parse_solver(os.path.join(CONFIGS, "test_resources", "caffenet_solver.prototxt"))
    assert t.param_count == 60965224 - 4097000 + 8194 == 56876418 and t.batch_size == 4
    with pytest.raises(cos.CosError, match="clip_gradients"):  # LRCN: clipping + LSTM are off the accelerated path
        cos.parse_solver(os.path.join(CONFIGS, "data", "lrcn_solver.prototxt"))


def test_parser_rejects_what_is_off_the_path(cos, tmp_path):
    p = tmp_path / "s.prototxt"
    p.write_text('net: "nope.prototxt"\nbase_lr: 0.1\nlr_policy: "fixed"\n')
    with pytest.raises(cos.CosError, match="cannot read net file"):
        cos.parse_solver(str(p))
    p.write_text('type: "Adam"\nbase_lr: 0.1\nlr_policy: "fixed"\nnet_param { }\n')
    with pytest.raises(cos.CosError, match="only SGD"):
        cos.parse_solver(str(p))
    p.write_text('base_lr: 0.1 lr_policy: "fixed" net_param { layer { name: "x" type: "LSTM" bottom: "a" top: "b" } }')
    with pytest.raises(cos.CosError, match="not understood"):
        cos.parse_solver(str(p))
    with pytest.raises(cos.CosError, match="cannot read solver file"):
        cos.parse_solver(str(tmp_path / "missing.prototxt"))
    inp = ('net_param { layer { name: "d" type: "Input" top: "data" input_param { shape { dim: 1 dim: 1 dim: 4 dim: 4 } } } '
           'layer { name: "ip" type: "InnerProduct" bottom: "data" top: "ip" inner_product_param { num_output: 2 } } }')
    p.write_text('base_lr: 0.1 lr_policy: "fixed" regularization_type: "L1" ' + inp)
    assert cos.parse_solver(str(p)).regularization_type == "L1"     # sgd_solver.cpp:161-168, on the fused path
    p.write_text('base_lr: 0.1 lr_policy: "fixed" regularization_type: "L3" ' + inp)
    with pytest.raises(cos.CosError, match="Unknown regularization type"):
        cos.parse_solver(str(p))


@pytest.mark.skipif(gpu_count() > 0, reason="only meaningful on a GPU-less box")
def test_compute_fails_loudly_without_a_gpu(cos):
    d = cos.SolverDesc([100], lr_policy="fixed", base_lr=0.1)
    with pytest.raises(cos.CosError, match="no CPU path"):
        cos.CaffeNet(d)


def test_adapter_rejects_bogus_addresses(cos):
    # CaffeNetTest.connectbogus: {"0x222","0x333"} must not connect
    a = cos.PeerAdapter(2, 0)
    try:
        assert a.address().startswith("cosb200://")
        assert not a.connect(["0x222", "0x333"])
        assert not a.connect(["", "cosb200://1/cosb200-1-r1-deadbeefdeadbeef"])  # well-formed, nobody listening
    finally:
        a.close()


def test_adapter_loopback_two_ranks_in_process(cos):
    # two adapters in one process: connect, CTRL barrier, fd + metadata passing
    import threading
    ads = [cos.PeerAdapter(2, r) for r in range(2)]
    addrs = [a.address() for a in ads]
    res = [None, None]

    def run(r):
        ok = ads[r].connect(addrs)
        ok = ok and ads[r].barrier(5000)
        res[r] = ok

    th = [threading.Thread(target=run, args=(r,)) for r in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert res == [True, True]
    fd = os.memfd_create("cos_test")
    os.write(fd, b"hello peer memory")
    assert ads[0].offer_fd("blob", fd, b"meta-bytes")
    got, meta = ads[1].fetch_fd(0, "blob")
    assert got >= 0 and meta.startswith(b"meta-bytes")
    os.lseek(got, 0, os.SEEK_SET)
    assert os.read(got, 64) == b"hello peer memory"
    os.close(got)
    os.close(fd)
    with pytest.raises(cos.CosError, match="not offered"):
        ads[1].fetch_fd(0, "never-offered", timeout_ms=200)
    [a.close() for a in ads]


def test_jni_shim_type_checks_and_covers_the_18_natives():
    """Without a JDK, the JNI shim is type-checked against a stand-in jni.h and
    must define one Java_com_yahoo_ml_jcaffe_CaffeNet_* export per native the
    reference's CaffeNet.java declares (CaffeNet.java:60-230; the list is stored
    in tests/golden/reference_interfaces.json)."""
    import subprocess
    src = os.path.join(ROOT, "caffeonspark_b200", "csrc", "jni_shim.cpp")
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-Werror", "-I",
                        os.path.join(ROOT, "tests", "jni_stub"), src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    natives = ["allocate", "deallocate", "connect", "sync", "init", "predict", "train", "localAddresses", "deviceID",
               "getInitIter", "getMaxIter", "getTestIter", "getTestInterval", "snapshot",
               "getValidationOutputBlobNames", "getValidationOutputBlobs", "validation", "aggregateValidationOutputs"]
    text = open(src).read()
    for n in natives:
        assert f"Java_com_yahoo_ml_jcaffe_CaffeNet_{n}(" in text, n
    with open(os.path.join(ROOT, "tests", "golden", "reference_interfaces.json")) as f:
        declared = set(json.load(f)["caffenet_java_natives"])
    assert declared == set(natives), declared ^ set(natives)


def test_every_entry_point_survives_null_and_invalid_arguments(cos):
    """Error behaviour at the boundary: a NULL handle / NULL pointers must come back as the failure value
    (0 / -1 / NULL) with an error string -- never a crash (the JVM would die with the executor)."""
    from caffeonspark_b200 import _lib
    L = _lib.lib()
    N = None
    assert L.cos_net_local_addresses(N, None) == -1
    assert L.cos_net_connect(N, None, 0) == 0
    assert L.cos_net_sync(N) == 0
    assert L.cos_net_init(N, 0, 1) == 0
    assert L.cos_net_train(N, 0, None, 0) == 0
    assert L.cos_net_predict(N, 0, None, 0, None, 0, None) == -1
    assert L.cos_net_validation(N, None, 0) == 0
    assert L.cos_net_aggregate_validation_outputs(N) == 0
    for fn in (L.cos_net_device_id, L.cos_net_get_init_iter, L.cos_net_get_max_iter, L.cos_net_get_test_iter):
        assert fn(N, 0) == -1 and fn(N, -1) == -1
    assert L.cos_net_get_test_interval(N) == -1
    assert L.cos_net_snapshot(N) == -1
    assert L.cos_net_snapshot_filename(N, 0, 0, None, 0) == 0
    assert L.cos_net_get_validation_output_blob_names(N, None) == -1
    assert L.cos_net_get_validation_output_blobs(N, 1, None) == -1
    assert L.cos_net_set_forward_backward(N, _lib.FORWARD_BACKWARD_FN(), None) == 0
    assert L.cos_net_data(N, 0) is None and L.cos_net_diff(N, 0) is None and L.cos_net_history(N, 0) is None
    assert L.cos_net_param_count(N) == -1
    assert L.cos_net_shard(N, 0, None, None) == 0
    assert L.cos_net_iter(N) == -1
    assert L.cos_net_learning_rate(N) == 0.0 and L.cos_net_last_loss(N) == 0.0
    assert L.cos_net_sync_step(N, 0, None) == 0
    assert L.cos_net_all_gather_weights(N, 0, None) == 0
    assert L.cos_net_synchronize(N) == 0
    assert L.cos_net_set_option(N, b"grid", 1) == 0 and L.cos_net_get_option(N, b"grid") == -1
    assert L.cos_net_last_kernel_ms(N) == -1.0 and L.cos_net_launch_count(N) == 0
    L.cos_net_deallocate(N)
    out = ctypes.c_void_p()
    assert L.cos_net_allocate(None, None, None, 1, 1, 0, 1, 0, -1, 0, ctypes.byref(out)) == 0
    assert b"solver_conf_file" in L.cos_last_error()
    assert L.cos_net_allocate(b"/nonexistent.prototxt", b"", b"", 1, 1, 0, 1, 0, -1, 0, ctypes.byref(out)) == 0
    assert L.cos_net_allocate_desc(None, 1, 1, 0, 1, 0, -1, ctypes.byref(out)) == 0
    assert L.cos_net_allocate_desc(None, 1, 1, 0, 1, 0, -1, None) == 0
    # adapter
    assert L.cos_adapter_create(0, 0) is None and L.cos_adapter_create(2, 5) is None
    assert L.cos_adapter_address(N) == b""
    assert L.cos_adapter_connect(N, None, 0) == 0 and L.cos_adapter_barrier(N, 10) == 0
    assert L.cos_adapter_offer_fd(N, b"k", -1, None, 0) == 0
    assert L.cos_adapter_fetch_fd(N, 0, b"k", None, 0, 10) == -2
    L.cos_adapter_destroy(N)
    # pure helpers
    assert L.cos_learning_rate(None, 0.1, 0.0, 0.0, 1, None, 0, 1, 0, None) == -1.0
    assert L.cos_parse_solver(None, None, None, None, None, 0, None, None, 0, None, 0, None) == -1
    assert L.cos_caffemodel_write(None, None, 0, None, None, None, None, None) == 0
    assert L.cos_caffemodel_read(None, None, 0, None, 0) == -1
    assert L.cos_solverstate_write(None, 0, 0, None, 0, None, None, None) == 0
    assert L.cos_solverstate_read(None, None, None, None, 0, -1, None, 0) == -1


def test_prototxt_parser_never_crashes_on_mutated_input(cos, tmp_path):
    """Fuzz: truncations and byte flips of a valid net definition must parse or fail with an error, never crash."""
    from caffeonspark_b200 import nets
    rng = np.random.RandomState(3)
    base = nets.net_prototxt("cifar10_quick")
    solver = tmp_path / "s.prototxt"
    netf = tmp_path / "n.prototxt"
    solver.write_text('net: "n.prototxt"\nbase_lr: 0.01\nlr_policy: "fixed"\n')
    ok = bad = 0
    for trial in range(300):
        b = bytearray(base.encode())
        kind = trial % 3
        if kind == 0:
            b = b[:rng.randint(0, len(b))]
        elif kind == 1:
            for _ in range(rng.randint(1, 6)):
                b[rng.randint(0, len(b))] = rng.randint(32, 127)
        else:
            i, j = sorted(rng.randint(0, len(b), 2))
            del b[i:j]
        netf.write_bytes(bytes(b))
        try:
            d = cos.parse_solver(str(solver))
            assert all(c >= 0 for c in d.counts)
            ok += 1
        except cos.CosError:
            bad += 1
    assert ok + bad == 300 and bad > 0


def test_parser_rejects_degenerate_geometry(cos, tmp_path):
    head = ('layer { name: "d" type: "Input" top: "data" input_param { shape { dim: 2 dim: 4 dim: 8 dim: 8 } } }\n')
    bad = ['layer { name: "c" type: "Convolution" bottom: "data" top: "c" convolution_param { num_output: 4 kernel_size: 3 stride: 0 } }',
           'layer { name: "c" type: "Convolution" bottom: "data" top: "c" convolution_param { num_output: 4 kernel_size: 3 group: 3 } }',
           'layer { name: "c" type: "Convolution" bottom: "data" top: "c" convolution_param { num_output: 4 kernel_size: 3 dilation: 0 } }',
           'layer { name: "p" type: "Pooling" bottom: "data" top: "p" pooling_param { kernel_size: 2 stride: 0 } }',
           'layer { name: "i" type: "InnerProduct" bottom: "data" top: "i" inner_product_param { num_output: 0 } }']
    solver = tmp_path / "s.prototxt"
    for layer in bad:
        solver.write_text('base_lr: 0.1 lr_policy: "fixed" net_param { ' + head + layer + ' }')
        with pytest.raises(cos.CosError, match="bad "):
            cos.parse_solver(str(solver))
    solver.write_text('base_lr: 0.1 lr_policy: "fixed" net_param { ' + head +
                      'layer { name: "c" type: "Convolution" bottom: "data" top: "c" convolution_param '
                      '{ num_output: 6 kernel_h: 3 kernel_w: 2 stride_h: 2 pad_w: 1 group: 2 bias_term: false } } }')
    d = cos.parse_solver(str(solver))
    assert d.counts == [6 * 2 * 3 * 2]


def test_gradient_producer_modules_match_the_flat_layout():
    """The PyTorch stand-in for Net::ForwardBackward must expose its parameters in learnable_params() order with
    exactly the blob sizes of the flat Params buffer (SURVEY App. D), or aliasing data_/diff_ would be wrong."""
    from caffeonspark_b200 import nets
    for name, P in nets.EXPECTED_PARAM_COUNT.items():
        counts, lm, dm, names = nets.layout(name)
        mod = nets.torch_module(name)
        sizes = [p.numel() for p in mod.parameters()]
        assert sizes == counts and sum(sizes) == P, name
        assert len(lm) == len(dm) == len(names) == len(counts)
        # Caffe blob shapes == torch parameter shapes (conv: [out, in/g, kh, kw]; ip: [out, in]; bias: [out])
        import torch
        c, h, w = nets.NETS[name]["input"]
        if name != "caffenet":  # a CPU forward/backward of the two small nets proves the module is well-formed
            x = torch.rand(2, c, h, w)
            loss = torch.nn.CrossEntropyLoss()(mod(x), torch.tensor([1, 3]))
            loss.backward()
            assert all(p.grad is not None and p.grad.shape == p.shape for p in mod.parameters())


def test_adapter_barrier_times_out_when_a_peer_never_arrives(cos):
    """Failure detection on the control plane: the reference blocks forever in BlockingQueue::pop when a peer
    dies (SURVEY section 5); here the barrier returns false after its time-out and fetches fail cleanly when
    the peer has gone away."""
    import time
    a, b = cos.PeerAdapter(2, 0), cos.PeerAdapter(2, 1)
    addrs = [a.address(), b.address()]
    import threading
    oks = [None, None]
    th = [threading.Thread(target=lambda r=r, ad=ad: oks.__setitem__(r, ad.connect(addrs))) for r, ad in enumerate((a, b))]
    [t.start() for t in th]
    [t.join() for t in th]
    assert oks == [True, True]
    t0 = time.time()
    assert a.barrier(300) is False            # rank 1 never calls barrier()
    assert 0.25 < time.time() - t0 < 5.0
    assert "timed out" in cos.caffenet._err()
    assert b.barrier(2000) is True            # ... the token rank 0 sent is still counted: b completes
    b.close()                                 # peer goes away
    with pytest.raises(cos.CosError):
        a.fetch_fd(1, "anything", timeout_ms=300)
    a.close()


def test_bench_algorithmic_byte_model_matches_design():
    """bench.py's roofline numerators are the formulas of DESIGN.md section 4."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    # importing bench.py redirects fd 1; only load the function's source instead
    src = open(os.path.join(ROOT, "bench.py")).read()
    start = src.index("def algorithmic_bytes")
    end = min(src.index("\ndef ", start + 10), src.index("\nclass ", start + 10))
    ns = {}
    exec(src[start:end], ns)
    f = ns["algorithmic_bytes"]
    P = 60965224
    assert f(P, 1, 0, 1, False) == (24 * P, 0)
    assert f(P, 1, 0, 0, False) == (20 * P, 0)
    hbm, nvl = f(P, 8, 1, 1, False)
    assert nvl == pytest.approx(8 * P * 7 / 8)                   # (b_g + 4) * P * (N-1)/N, b_g = 4
    assert f(P, 8, 1, 1, True)[1] == pytest.approx(6 * P * 7 / 8)  # bf16 wire
    assert f(P, 4, 2, 1, False)[1] == 4 * P * 3                   # one-shot pulls (N-1) full gradients
    assert f(P, 8, 1, 1, False, nvls=True)[1] == pytest.approx(4 * P * 9 / 8)   # NVLS: 4P(1 + 1/N)
    assert f(P, 8, 1, 1, True, push=True)[1] == pytest.approx(6 * P * 7 / 8)    # push: same wire bytes as pull
    assert f(P, 8, 1, 1, True, push=True)[0] < f(P, 8, 1, 1, True)[0]           # ... without the cast pre-pass
    assert spec is not None


@pytest.fixture
def sock_dir():
    """A fresh directory with a short path: a socket path must fit sun_path (108 bytes), which pytest's tmp_path
    under a deep $TMPDIR does not."""
    import pathlib
    import shutil
    import tempfile
    d = tempfile.mkdtemp(prefix="cos", dir="/tmp")
    yield pathlib.Path(d)
    shutil.rmtree(d, ignore_errors=True)


def test_adapter_pathname_sockets_for_separate_containers(cos, sock_dir, monkeypatch):
    """COS_SOCKET_DIR: endpoints become socket files in a shared directory (executors that do not share a network
    namespace cannot see each other's abstract sockets); same protocol, files removed on close."""
    import threading
    monkeypatch.setenv("COS_SOCKET_DIR", str(sock_dir))
    ads = [cos.PeerAdapter(2, r) for r in range(2)]
    addrs = [a.address() for a in ads]
    assert all(a.startswith("cosb200://") and str(sock_dir) in a and a.endswith(".sock") for a in addrs)
    assert len(list(sock_dir.glob("*.sock"))) == 2
    oks = [None, None]
    th = [threading.Thread(target=lambda r=r: oks.__setitem__(r, ads[r].connect(addrs) and ads[r].barrier(5000)))
          for r in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert oks == [True, True]
    fd = os.memfd_create("x")
    os.write(fd, b"payload")
    ads[1].offer_fd("k", fd, b"m")
    got, meta = ads[0].fetch_fd(1, "k")
    os.lseek(got, 0, os.SEEK_SET)
    assert os.read(got, 16) == b"payload" and meta.startswith(b"m")
    os.close(got)
    os.close(fd)
    [a.close() for a in ads]
    assert list(sock_dir.glob("*.sock")) == []
    monkeypatch.delenv("COS_SOCKET_DIR")
    a = cos.PeerAdapter(2, 0)
    assert not a.connect(["", "cosb200://1/" + str(sock_dir) + "/cosb200-1-r1-00.sock"])  # nobody there
    assert not a.connect(["", "cosb200://1//etc/passwd"])                                   # not one of ours
    a.close()
