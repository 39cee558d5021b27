"""Python mirror of ``com.yahoo.ml.jcaffe.CaffeNet`` over the C ABI.

Reference: caffe-distri/src/main/java/com/yahoo/ml/jcaffe/CaffeNet.java:20-232
(public API, same method names and argument meaning) and
caffe-distri/src/main/cpp/jni/JniCaffeNet.cpp (failure conventions).  Used by
the tests (which read like CaffeNetTest.java) and by the benchmark harness in
the role ``CaffeProcessor`` plays on the Scala side.
"""
import ctypes

from . import _lib
from ._lib import FORWARD_BACKWARD_FN, cos_blob, cos_solver_desc


class CosError(RuntimeError):
    """What the JNI shim would raise as java.lang.Exception / RuntimeException."""


def _err():
    return _lib.lib().cos_last_error().decode("utf-8", "replace")


def chunk(param_count, cluster_size, peer):
    """SocketSync::chunk (socket_sync_cpu.cpp:46-54) -> (offset, size) in elements."""
    o, s = ctypes.c_uint64(), ctypes.c_uint64()
    _lib.lib().cos_chunk(param_count, cluster_size, peer, ctypes.byref(o), ctypes.byref(s))
    return o.value, s.value


def learning_rate(lr_policy, base_lr, gamma=0.0, power=0.0, stepsize=1, stepvalues=(), max_iter=1, it=0,
                  current_step=0):
    """SGDSolver::GetLearningRate (sgd_solver.cpp:27-63); returns (rate, current_step)."""
    sv = (ctypes.c_int * max(1, len(stepvalues)))(*stepvalues)
    step = ctypes.c_int(current_step)
    r = _lib.lib().cos_learning_rate(lr_policy.encode(), base_lr, gamma, power, int(stepsize), sv, len(stepvalues),
                                     int(max_iter), int(it), ctypes.byref(step))
    if r < 0:
        raise CosError(_err())
    return r, step.value


class SolverDesc:
    """Solver hyper-parameters + learnable blob layout (cos_solver_desc)."""

    def __init__(self, counts, lr_mult=None, decay_mult=None, lr_policy="fixed", base_lr=0.01, gamma=0.0, power=0.0,
                 stepsize=1, stepvalues=(), max_iter=0, momentum=0.0, weight_decay=0.0, test_iter=0,
                 test_interval=0, snapshot_prefix="", grad_dtype="fp32", init_iter=0, batch_size=0,
                 regularization_type="L2", type="SGD", delta=1e-8, rms_decay=0.0):
        self.counts = [int(c) for c in counts]
        self.lr_mult = [float(x) for x in (lr_mult if lr_mult is not None else [1.0] * len(self.counts))]
        self.decay_mult = [float(x) for x in (decay_mult if decay_mult is not None else [1.0] * len(self.counts))]
        self.lr_policy, self.base_lr, self.gamma, self.power = lr_policy, base_lr, gamma, power
        self.stepsize, self.stepvalues, self.max_iter = stepsize, tuple(stepvalues), max_iter
        self.momentum, self.weight_decay = momentum, weight_decay
        self.test_iter, self.test_interval, self.snapshot_prefix = test_iter, test_interval, snapshot_prefix
        self.grad_dtype, self.init_iter, self.batch_size = grad_dtype, init_iter, batch_size
        self.regularization_type = regularization_type
        self.type, self.delta, self.rms_decay = type, delta, rms_decay  # SolverParameter.type / delta / rms_decay

    @property
    def param_count(self):
        return max(1, sum(self.counts))

    def hyper(self):
        """Keyword arguments understood by oracle.Simulation / run_ref_*."""
        return dict(lr_policy=self.lr_policy, base_lr=self.base_lr, gamma=self.gamma, power=self.power,
                    stepsize=self.stepsize, stepvalues=self.stepvalues, max_iter=self.max_iter,
                    momentum=self.momentum, weight_decay=self.weight_decay,
                    regularization_type=self.regularization_type)

    def to_c(self):
        n = len(self.counts)
        keep = dict(counts=(ctypes.c_int64 * max(1, n))(*self.counts),
                    lr=(ctypes.c_float * max(1, n))(*self.lr_mult),
                    dm=(ctypes.c_float * max(1, n))(*self.decay_mult),
                    sv=(ctypes.c_int * max(1, len(self.stepvalues)))(*self.stepvalues),
                    pol=self.lr_policy.encode(), pre=self.snapshot_prefix.encode(), typ=self.type.encode())
        d = cos_solver_desc()
        d.nblobs, d.counts, d.lr_mult, d.decay_mult = n, keep["counts"], keep["lr"], keep["dm"]
        d.lr_policy, d.base_lr, d.gamma, d.power = keep["pol"], self.base_lr, self.gamma, self.power
        d.stepsize, d.stepvalues, d.nstepvalues = int(self.stepsize), keep["sv"], len(self.stepvalues)
        d.max_iter, d.momentum, d.weight_decay = int(self.max_iter), self.momentum, self.weight_decay
        d.test_iter, d.test_interval, d.snapshot_prefix = int(self.test_iter), int(self.test_interval), keep["pre"]
        d.grad_dtype = 1 if self.grad_dtype == "bf16" else 0
        d.init_iter = int(self.init_iter)
        d.regularization_l1 = 1 if self.regularization_type == "L1" else 0
        d.type, d.delta, d.rms_decay = keep["typ"], self.delta, self.rms_decay
        return d, keep


def parse_solver(solver_conf_file):
    """Utils.GetSolverParam + the learnable layout of the net it names."""
    L = _lib.lib()
    cap = 4096
    d = cos_solver_desc()
    c, lm, dm = (ctypes.c_int64 * cap)(), (ctypes.c_float * cap)(), (ctypes.c_float * cap)()
    pol, pre = ctypes.create_string_buffer(256), ctypes.create_string_buffer(256)
    sv, bs = (ctypes.c_int * 64)(), ctypes.c_int()
    n = L.cos_parse_solver(str(solver_conf_file).encode(), ctypes.byref(d), c, lm, dm, cap, pol, pre, 256, sv, 64,
                           ctypes.byref(bs))
    if n < 0:
        raise CosError(_err())
    return SolverDesc(list(c[:n]), list(lm[:n]), list(dm[:n]), lr_policy=pol.value.decode(), base_lr=d.base_lr,
                      gamma=d.gamma, power=d.power, stepsize=d.stepsize, stepvalues=list(sv[:d.nstepvalues]),
                      max_iter=d.max_iter, momentum=d.momentum, weight_decay=d.weight_decay, test_iter=d.test_iter,
                      test_interval=d.test_interval, snapshot_prefix=pre.value.decode(), batch_size=bs.value,
                      regularization_type="L1" if d.regularization_l1 else "L2", type=d.type.decode(), delta=d.delta,
                      rms_decay=d.rms_decay)


def read_caffemodel_blob(path, layer_name, blob_index=0):
    """One blob of a Caffe .caffemodel (ours or stock Caffe's) as a flat float32 numpy array."""
    import numpy as np
    L = _lib.lib()
    n = L.cos_caffemodel_read(str(path).encode(), layer_name.encode(), blob_index, None, 0)
    if n < 0:
        raise CosError(_err())
    out = np.empty(n, np.float32)
    L.cos_caffemodel_read(str(path).encode(), layer_name.encode(), blob_index, out.ctypes.data, n)
    return out


def read_solverstate(path):
    """-> (iter, current_step, learned_net, [history blobs as flat float32 arrays]) of a Caffe .solverstate."""
    import numpy as np
    L = _lib.lib()
    it, step = ctypes.c_int(), ctypes.c_int()
    buf = ctypes.create_string_buffer(4096)
    n = L.cos_solverstate_read(str(path).encode(), ctypes.byref(it), ctypes.byref(step), buf, 4096, -1, None, 0)
    if n < 0:
        raise CosError(_err())
    hist = []
    for k in range(n):
        m = L.cos_solverstate_read(str(path).encode(), None, None, None, 0, k, None, 0)
        a = np.empty(m, np.float32)
        L.cos_solverstate_read(str(path).encode(), None, None, None, 0, k, a.ctypes.data, m)
        hist.append(a)
    return it.value, step.value, buf.value.decode(), hist


class _DevArray:
    """__cuda_array_interface__ view of a raw device pointer (zero-copy)."""

    def __init__(self, ptr, n, typestr="<f4"):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 3, "strides": None}


def _blob_array(data):
    """list of host arrays (numpy float32 / CPU torch float32, up to 4-D) -> cos_blob[]"""
    blobs = (cos_blob * max(1, len(data)))()
    keep = []
    for i, a in enumerate(data):
        if hasattr(a, "data_ptr"):  # torch CPU tensor (pinned or not)
            if a.is_cuda or str(a.dtype) != "torch.float32" or not a.is_contiguous():
                raise CosError("train(): blobs must be contiguous float32 HOST tensors")
            ptr, shape = a.data_ptr(), tuple(a.shape)
        else:
            import numpy as np
            a = np.ascontiguousarray(a, dtype=np.float32)
            ptr, shape = a.ctypes.data, a.shape
        keep.append(a)
        shape = tuple(shape) + (1,) * (4 - len(shape))
        blobs[i].data, blobs[i].num, blobs[i].channels, blobs[i].height, blobs[i].width = ptr, *[int(s) for s in shape]
    return blobs, keep


class CaffeNet:
    """Same surface as com.yahoo.ml.jcaffe.CaffeNet (CaffeNet.java)."""

    NONE, RDMA, SOCKET = 0, 1, 2  # CaffeNet.java:21-23

    def __init__(self, solver_conf_file, input_model_file="", input_state_file="", num_local_devices=1,
                 cluster_size=1, node_rank=0, isTraining=True, connection_type=0, start_device_id=-1,
                 validation_net_id=0):
        """CaffeNet.java:44-58.  `solver_conf_file` is a prototxt path or a SolverDesc."""
        self._L = _lib.lib()
        self._h = ctypes.c_void_p()
        self._fb_keep = None
        self.cluster_size, self.node_rank, self.num_local_devices = cluster_size, node_rank, num_local_devices
        if isinstance(solver_conf_file, SolverDesc):
            self.desc = solver_conf_file
            d, keep = self.desc.to_c()
            ok = self._L.cos_net_allocate_desc(ctypes.byref(d), num_local_devices, cluster_size, node_rank,
                                               int(bool(isTraining)), connection_type, start_device_id,
                                               ctypes.byref(self._h))
            del keep
        else:
            self.desc = parse_solver(solver_conf_file)  # Utils.GetSolverParam (CaffeNet.java:53)
            ok = self._L.cos_net_allocate(str(solver_conf_file).encode(), (input_model_file or "").encode(),
                                          (input_state_file or "").encode(), num_local_devices, cluster_size,
                                          node_rank, int(bool(isTraining)), connection_type, start_device_id,
                                          validation_net_id, ctypes.byref(self._h))
        if not ok:
            self._h = ctypes.c_void_p()
            raise CosError("Failed to create CaffeNet object: " + _err())  # CaffeNet.java:54-57

    # ---- BaseObject.java:36-49
    def deallocate(self):
        if self._h:
            self._L.cos_net_deallocate(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.deallocate()
        except Exception:
            pass

    # ---- the JNI natives
    def localAddresses(self):
        arr = ctypes.POINTER(ctypes.c_char_p)()
        n = self._L.cos_net_local_addresses(self._h, ctypes.byref(arr))
        if n < 0:
            return None
        return [arr[i].decode() for i in range(n)]

    def connect(self, addresses):
        if addresses is None:
            return bool(self._L.cos_net_connect(self._h, None, 0))
        arr = (ctypes.c_char_p * max(1, len(addresses)))(*[None if a is None else a.encode() for a in addresses])
        return bool(self._L.cos_net_connect(self._h, arr, len(addresses)))

    def sync(self):
        return bool(self._L.cos_net_sync(self._h))

    def init(self, solver_index, enableNN=False):
        return bool(self._L.cos_net_init(self._h, solver_index, int(enableNN)))

    def train(self, solver_index, data):
        """One Solver::Step.  data=None raises like the JNI layer (JniCaffeNet.cpp:391-395)."""
        if data is None:
            self._L.cos_net_train(self._h, solver_index, None, 0)
            raise CosError(_err())
        blobs, keep = _blob_array(data)
        ok = bool(self._L.cos_net_train(self._h, solver_index, blobs, len(data)))
        del keep
        return ok

    def predict(self, solver_index, data, output_blobnames):
        return None  # forward-only inference is outside the sync library (cos_net_predict fails)

    def deviceID(self, solver_index):
        return self._L.cos_net_device_id(self._h, solver_index)

    def getInitIter(self, solver_index):
        return self._L.cos_net_get_init_iter(self._h, solver_index)

    def getMaxIter(self, solver_index):
        return self._L.cos_net_get_max_iter(self._h, solver_index)

    def getTestIter(self, solver_index):
        return self._L.cos_net_get_test_iter(self._h, solver_index)

    def getTestInterval(self):
        return self._L.cos_net_get_test_interval(self._h)

    def snapshot(self):
        return self._L.cos_net_snapshot(self._h)

    def snapshotFilename(self, it, isState):
        """CaffeNet.java:192-207: <snapshot_prefix>_iter_<it>.solverstate / .caffemodel (+ ".h5")."""
        if it < 0:
            return None
        buf = ctypes.create_string_buffer(4096)
        if not self._L.cos_net_snapshot_filename(self._h, it, int(bool(isState)), buf, 4096):
            return None
        return buf.value.decode()

    # ---- hot-path surface (what a native gradient producer uses)
    def last_error(self):
        return _err()

    def set_forward_backward(self, fn):
        """fn(solver_index, blobs:[(dev_ptr, (n,c,h,w))], loss_dev_ptr, stream_ptr) -> 0/None on success."""
        def tramp(user, solver_index, blobs, n, loss_dev, stream):
            try:
                ins = [(blobs[i].data, (blobs[i].num, blobs[i].channels, blobs[i].height, blobs[i].width))
                       for i in range(n)]
                rc = fn(solver_index, ins, loss_dev, stream)
                return int(rc or 0)
            except Exception:  # never unwind through C
                import traceback
                traceback.print_exc()
                return 1
        self._fb_keep = FORWARD_BACKWARD_FN(tramp)
        return bool(self._L.cos_net_set_forward_backward(self._h, self._fb_keep, None))

    def param_count(self):
        return self._L.cos_net_param_count(self._h)

    def data_ptr(self, solver_index=0):
        return self._L.cos_net_data(self._h, solver_index)

    def diff_ptr(self, solver_index=0):
        return self._L.cos_net_diff(self._h, solver_index)

    def history_ptr(self, solver_index=0):
        return self._L.cos_net_history(self._h, solver_index)

    def update_history_ptr(self, solver_index=0):
        return self._L.cos_net_update_history(self._h, solver_index)

    def _torch_view(self, ptr, solver_index=0):
        import torch
        return torch.as_tensor(_DevArray(ptr, self.param_count()), device=f"cuda:{self.deviceID(solver_index)}")

    def data(self, solver_index=0):
        """Zero-copy torch view of Params::data_ (flat fp32 weights) of local solver `solver_index`."""
        return self._torch_view(self.data_ptr(solver_index), solver_index)

    def diff(self, solver_index=0):
        return self._torch_view(self.diff_ptr(solver_index), solver_index)

    def history(self, solver_index=0):
        return self._torch_view(self.history_ptr(solver_index), solver_index)

    def update_history(self, solver_index=0):
        """AdaDelta's second history (history of updates) as a torch view; None for the other solvers."""
        ptr = self.update_history_ptr(solver_index)
        return self._torch_view(ptr, solver_index) if ptr else None

    def global_rank(self, solver_index=0):
        """Rank of local solver `solver_index` in the collective of cluster_size x num_local_devices ranks."""
        return self.node_rank * self.num_local_devices + solver_index

    def shard(self, rank=None):
        o, s = ctypes.c_uint64(), ctypes.c_uint64()
        if not self._L.cos_net_shard(self._h, self.global_rank(0) if rank is None else rank, ctypes.byref(o),
                                     ctypes.byref(s)):
            raise CosError(_err())
        return o.value, s.value

    def iter(self):
        return self._L.cos_net_iter(self._h)

    def learning_rate(self):
        return self._L.cos_net_learning_rate(self._h)

    def last_loss(self):
        return self._L.cos_net_last_loss(self._h)

    def sync_step(self, solver_index=0, stream=None):
        return bool(self._L.cos_net_sync_step(self._h, solver_index, stream))

    def all_gather_weights(self, solver_index=0, stream=None):
        return bool(self._L.cos_net_all_gather_weights(self._h, solver_index, stream))

    def synchronize(self):
        return bool(self._L.cos_net_synchronize(self._h))

    def set_option(self, name, value):
        if not self._L.cos_net_set_option(self._h, name.encode(), int(value)):
            raise CosError(_err())

    def get_option(self, name):
        return self._L.cos_net_get_option(self._h, name.encode())

    def last_kernel_ms(self):
        return self._L.cos_net_last_kernel_ms(self._h)

    def launch_count(self):
        return self._L.cos_net_launch_count(self._h)

    def fill(self, which, seed, stream, amp, solver_index=0):
        """Seeded synthetic fill of data_ / diff_ / history on the device (same generator as the oracle's)."""
        k = {"data": 0, "diff": 1, "history": 2}.get(which, which)
        if not self._L.cos_net_fill(self._h, solver_index, int(k), int(seed), int(stream), float(amp)):
            raise CosError(_err())


class PeerAdapter:
    """cos_adapter: the SocketAdapter/SocketChannel analogue (control plane only)."""

    def __init__(self, cluster_size, rank):
        self._L = _lib.lib()
        self._a = self._L.cos_adapter_create(cluster_size, rank)
        if not self._a:
            raise CosError(_err())

    def close(self):
        if self._a:
            self._L.cos_adapter_destroy(self._a)
            self._a = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def address(self):
        return self._L.cos_adapter_address(self._a).decode()

    def connect(self, addresses):
        arr = (ctypes.c_char_p * max(1, len(addresses)))(*[None if a is None else a.encode() for a in addresses])
        return bool(self._L.cos_adapter_connect(self._a, arr, len(addresses)))

    def barrier(self, timeout_ms=10000):
        return bool(self._L.cos_adapter_barrier(self._a, timeout_ms))

    def offer_fd(self, key, fd, meta=b""):
        buf = ctypes.create_string_buffer(meta, len(meta)) if meta else None
        return bool(self._L.cos_adapter_offer_fd(self._a, key.encode(), fd, buf, len(meta)))

    def fetch_fd(self, peer, key, meta_cap=256, timeout_ms=10000):
        """-> (fd or -1, meta bytes); raises CosError when the peer never offered `key`."""
        buf = ctypes.create_string_buffer(meta_cap)
        fd = self._L.cos_adapter_fetch_fd(self._a, peer, key.encode(), buf, meta_cap, timeout_ms)
        if fd == -2:
            raise CosError(_err())
        return fd, buf.raw
