"""CPU tests of the hand-rolled Caffe binaryproto reader/writer (snapshot files)
against the REAL protobuf runtime: message classes are built at run time from a
descriptor of the caffe.proto subset the snapshots use, so encoding and decoding
are checked by an independent implementation.  The field numbers of that
descriptor are verified against those of the reference's caffe.proto, stored in
tests/golden/reference_interfaces.json."""
import ctypes
import json
import os

import numpy as np
import pytest

from google.protobuf import descriptor_pb2, descriptor_pool, message_factory

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_interfaces.json")
F = descriptor_pb2.FieldDescriptorProto

SUBSET = {  # message -> [(name, number, type, label, type_name, packed)]
    "BlobShape": [("dim", 1, F.TYPE_INT64, F.LABEL_REPEATED, None, True)],
    "BlobProto": [("num", 1, F.TYPE_INT32, F.LABEL_OPTIONAL, None, False),
                  ("channels", 2, F.TYPE_INT32, F.LABEL_OPTIONAL, None, False),
                  ("height", 3, F.TYPE_INT32, F.LABEL_OPTIONAL, None, False),
                  ("width", 4, F.TYPE_INT32, F.LABEL_OPTIONAL, None, False),
                  ("data", 5, F.TYPE_FLOAT, F.LABEL_REPEATED, None, True),
                  ("shape", 7, F.TYPE_MESSAGE, F.LABEL_OPTIONAL, ".caffe.BlobShape", False)],
    "LayerParameter": [("name", 1, F.TYPE_STRING, F.LABEL_OPTIONAL, None, False),
                       ("type", 2, F.TYPE_STRING, F.LABEL_OPTIONAL, None, False),
                       ("bottom", 3, F.TYPE_STRING, F.LABEL_REPEATED, None, False),
                       ("blobs", 7, F.TYPE_MESSAGE, F.LABEL_REPEATED, ".caffe.BlobProto", False),
                       ("phase", 10, F.TYPE_INT32, F.LABEL_OPTIONAL, None, False)],
    "NetParameter": [("name", 1, F.TYPE_STRING, F.LABEL_OPTIONAL, None, False),
                     ("force_backward", 5, F.TYPE_BOOL, F.LABEL_OPTIONAL, None, False),
                     ("layer", 100, F.TYPE_MESSAGE, F.LABEL_REPEATED, ".caffe.LayerParameter", False)],
    "SolverState": [("iter", 1, F.TYPE_INT32, F.LABEL_OPTIONAL, None, False),
                    ("learned_net", 2, F.TYPE_STRING, F.LABEL_OPTIONAL, None, False),
                    ("history", 3, F.TYPE_MESSAGE, F.LABEL_REPEATED, ".caffe.BlobProto", False),
                    ("current_step", 4, F.TYPE_INT32, F.LABEL_OPTIONAL, None, False)],
}


@pytest.fixture(scope="module")
def pb():
    fdp = descriptor_pb2.FileDescriptorProto(name="caffe_subset_for_tests.proto", package="caffe", syntax="proto2")
    for msg, fields in SUBSET.items():
        m = fdp.message_type.add(name=msg)
        for name, number, typ, label, type_name, packed in fields:
            f = m.field.add(name=name, number=number, type=typ, label=label)
            if type_name:
                f.type_name = type_name
            if packed:
                f.options.packed = True
    pool = descriptor_pool.DescriptorPool()
    pool.Add(fdp)
    get = getattr(message_factory, "GetMessageClass", None)
    if get is None:  # older protobuf
        fac = message_factory.MessageFactory(pool)
        get = fac.GetPrototype
    return {n: get(pool.FindMessageTypeByName("caffe." + n)) for n in SUBSET}


def test_subset_field_numbers_match_reference_proto():
    with open(GOLD) as f:
        ref = json.load(f)["caffe_proto_fields"]
    for msg, fields in SUBSET.items():
        for name, number, *_ in fields:
            assert ref[msg].get(name) == number, (msg, name, number)


def _c_blobs(arrays):
    ptrs = (ctypes.c_void_p * len(arrays))(*[a.ctypes.data for a in arrays])
    nd = (ctypes.c_int * len(arrays))(*[a.ndim for a in arrays])
    dims = [d for a in arrays for d in a.shape]
    return ptrs, nd, (ctypes.c_int64 * len(dims))(*dims)


def _strs(xs):
    return (ctypes.c_char_p * len(xs))(*[x.encode() for x in xs])


def test_written_caffemodel_parses_with_real_protobuf(cos, pb, tmp_path):
    from caffeonspark_b200 import _lib
    L = _lib.lib()
    rng = np.random.RandomState(0)
    arrays = [rng.randn(20, 1, 5, 5).astype(np.float32), rng.randn(20).astype(np.float32),
              rng.randn(10, 300).astype(np.float32), rng.randn(10).astype(np.float32),
              rng.randn(3).astype(np.float32)]
    names = ["conv1", "conv1", "ip1", "ip1", "scale"]
    types = ["Convolution", "Convolution", "InnerProduct", "InnerProduct", "Bias"]
    ptrs, nd, dims = _c_blobs(arrays)
    path = str(tmp_path / "m.caffemodel")
    assert L.cos_caffemodel_write(path.encode(), b"LeNet", len(arrays), _strs(names), _strs(types), nd, dims, ptrs)
    net = pb["NetParameter"]()
    net.ParseFromString(open(path, "rb").read())
    assert net.name == "LeNet"
    assert [(l.name, l.type, len(l.blobs)) for l in net.layer] == [("conv1", "Convolution", 2),
                                                                    ("ip1", "InnerProduct", 2), ("scale", "Bias", 1)]
    flat = [b for l in net.layer for b in l.blobs]
    for a, b in zip(arrays, flat):
        assert list(b.shape.dim) == list(a.shape)
        assert np.array_equal(np.asarray(b.data, np.float32), a.ravel())
    # and our own reader
    out = np.empty(3000, np.float32)
    n = L.cos_caffemodel_read(path.encode(), b"ip1", 0, out.ctypes.data, out.size)
    assert n == 3000 and np.array_equal(out, arrays[2].ravel())
    assert L.cos_caffemodel_read(path.encode(), b"nope", 0, None, 0) == -1


def test_reads_caffemodel_written_by_real_protobuf(cos, pb, tmp_path):
    """What stock Caffe writes: extra fields we do not know (bottom, phase, force_backward), a blob with the
    legacy num/channels/height/width instead of shape, un-named layers without blobs."""
    from caffeonspark_b200 import _lib
    L = _lib.lib()
    rng = np.random.RandomState(1)
    net = pb["NetParameter"](name="n", force_backward=True)
    d = net.layer.add(name="data", type="MemoryData", phase=0)
    l1 = net.layer.add(name="conv1", type="Convolution", phase=0)
    l1.bottom.append("data")
    w = rng.randn(4, 3, 2, 2).astype(np.float32)
    b1 = l1.blobs.add(num=4, channels=3, height=2, width=2)  # legacy 4-D description
    b1.data.extend(w.ravel().tolist())
    bias = rng.randn(4).astype(np.float32)
    b2 = l1.blobs.add()
    b2.shape.dim.extend([4])
    b2.data.extend(bias.tolist())
    path = str(tmp_path / "stock.caffemodel")
    open(path, "wb").write(net.SerializeToString())
    out = np.empty(48, np.float32)
    assert L.cos_caffemodel_read(path.encode(), b"conv1", 0, out.ctypes.data, 48) == 48
    assert np.array_equal(out, w.ravel())
    assert L.cos_caffemodel_read(path.encode(), b"conv1", 1, out.ctypes.data, 48) == 4
    assert np.array_equal(out[:4], bias)
    assert L.cos_caffemodel_read(path.encode(), b"data", 0, None, 0) == -1  # layer exists, has no blobs
    assert d is not None


def test_solverstate_both_directions(cos, pb, tmp_path):
    from caffeonspark_b200 import _lib
    L = _lib.lib()
    rng = np.random.RandomState(2)
    hist = [rng.randn(6, 5).astype(np.float32), rng.randn(6).astype(np.float32)]
    ptrs, nd, dims = _c_blobs(hist)
    path = str(tmp_path / "s.solverstate")
    assert L.cos_solverstate_write(path.encode(), 1234, 3, b"/x/y_iter_1234.caffemodel", 2, nd, dims, ptrs)
    st = pb["SolverState"]()
    st.ParseFromString(open(path, "rb").read())
    assert (st.iter, st.current_step, st.learned_net) == (1234, 3, "/x/y_iter_1234.caffemodel")
    assert [list(h.shape.dim) for h in st.history] == [[6, 5], [6]]
    assert np.array_equal(np.asarray(st.history[0].data, np.float32), hist[0].ravel())
    # written by protobuf, read by us
    st2 = pb["SolverState"](iter=77, learned_net="m", current_step=2)
    hb = st2.history.add()
    hb.shape.dim.extend([3])
    hb.data.extend([1.5, -2.25, 3.0])
    p2 = str(tmp_path / "s2.solverstate")
    open(p2, "wb").write(st2.SerializeToString())
    it, step = ctypes.c_int(), ctypes.c_int()
    buf = ctypes.create_string_buffer(64)
    assert L.cos_solverstate_read(p2.encode(), ctypes.byref(it), ctypes.byref(step), buf, 64, -1, None, 0) == 1
    assert (it.value, step.value, buf.value) == (77, 2, b"m")
    out = np.empty(3, np.float32)
    assert L.cos_solverstate_read(p2.encode(), None, None, None, 0, 0, out.ctypes.data, 3) == 3
    assert out.tolist() == [1.5, -2.25, 3.0]


def test_garbage_is_rejected(cos, tmp_path):
    from caffeonspark_b200 import _lib
    L = _lib.lib()
    p = tmp_path / "junk.bin"
    p.write_bytes(bytes(range(256)) * 7)
    assert L.cos_caffemodel_read(str(p).encode(), b"x", 0, None, 0) == -1
    assert L.cos_solverstate_read(str(p).encode(), None, None, None, 0, -1, None, 0) == -1
    assert L.cos_caffemodel_read(str(tmp_path / "missing").encode(), b"x", 0, None, 0) == -1


def test_malformed_layer_is_an_error_not_a_partial_model(cos, pb, tmp_path):
    """A LayerParameter whose body is cut short must fail the whole read: returning the layers parsed so far would
    let a resume silently keep random weights for the rest (Net::CopyTrainedLayersFrom would have CHECK-failed)."""
    from caffeonspark_b200 import _lib
    L = _lib.lib()
    net = pb["NetParameter"](name="n")
    a = net.layer.add(name="a", type="InnerProduct")
    b = a.blobs.add()
    b.shape.dim.extend([2, 2])
    b.data.extend([1.0, 2.0, 3.0, 4.0])
    good = net.SerializeToString()
    bad_layer = b"\x0a\x01b" + b"\x12\x7f"  # name "b", then field 2 (type) announcing 127 bytes that are not there
    blob = good + b"\xa2\x06" + bytes([len(bad_layer)]) + bad_layer + good[2 + len("n"):]  # a, broken b, a again
    p = tmp_path / "broken.caffemodel"
    p.write_bytes(blob)
    assert L.cos_caffemodel_read(str(p).encode(), b"a", 0, None, 0) == -1
    assert b"malformed LayerParameter" in L.cos_last_error()
    p.write_bytes(good)
    assert L.cos_caffemodel_read(str(p).encode(), b"a", 0, None, 0) == 4
