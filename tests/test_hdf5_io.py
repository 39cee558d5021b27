"""CPU tests of the libhdf5-free HDF5 snapshot reader/writer (csrc/hdf5_io.cpp).

There is no libhdf5 / h5py in this environment, so the evidence is layered:
  1. the C++ READER is pinned on files libhdf5 itself wrote -- the reference's fixtures
     caffe-public/src/caffe/test/test_data/{solver_data,sample_data}.h5, stored under tests/golden/hdf5 --
     against (a) the raw bytes at the data offsets and (b) a second, independent mini-parser of the format
     written in Python below;
  2. the C++ WRITER's files are parsed by that Python mini-parser (not by the C++ reader alone), their message
     bytes are compared with the libhdf5-written ones, and they round-trip through the C++ reader;
  3. what the format cannot express here (chunked / gzip datasets) is rejected with a clear error.
What is NOT shown: libhdf5 opening the written files (no libhdf5 here)."""
import ctypes
import hashlib
import os
import struct

import numpy as np

FIX = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hdf5")


# ------------------------------------------------------------------ independent mini-parser (Python)
class MiniH5:
    """Walks superblock v0 -> v1 object headers -> group B-tree / local heap / symbol nodes; returns
    {path: dict(kind, shape, messages{type: bytes}, data(bytes))}."""

    def __init__(self, path):
        self.b = open(path, "rb").read()
        b = self.b
        assert b[:8] == b"\x89HDF\r\n\x1a\n" and b[8] == 0 and b[13] == 8 and b[14] == 8
        self.leaf_k, self.internal_k = struct.unpack_from("<HH", b, 16)
        self.eof = struct.unpack_from("<Q", b, 40)[0]
        self.objects = {}
        name_off, ohdr, cache = struct.unpack_from("<QQI", b, 56)
        self.root_cache = (cache, struct.unpack_from("<QQ", b, 80))
        self._object(ohdr, "")

    def _messages(self, addr):
        b = self.b
        ver, _, nmsg, ref, hsize = struct.unpack_from("<BBHII", b, addr)
        assert ver == 1 and ref == 1
        out, blocks = [], [(addr + 16, addr + 16 + hsize)]
        while blocks:
            pos, end = blocks.pop(0)
            while pos + 8 <= end and len(out) < nmsg:
                t, sz, fl = struct.unpack_from("<HHB", b, pos)
                assert sz % 8 == 0
                body = b[pos + 8:pos + 8 + sz]
                out.append((t, fl, body))
                if t == 0x10:
                    ca, cl = struct.unpack_from("<QQ", body)
                    blocks.append((ca, ca + cl))
                pos += 8 + sz
        assert len(out) == nmsg
        return out

    def _object(self, addr, path):
        b = self.b
        msgs = self._messages(addr)
        types = {t: (fl, body) for t, fl, body in msgs}
        if 0x11 in types:
            bt, hp = struct.unpack_from("<QQ", types[0x11][1])
            assert b[hp:hp + 4] == b"HEAP"
            dsize, free, daddr = struct.unpack_from("<QQQ", b, hp + 8)
            self.objects[path or "/"] = dict(kind="group", btree=bt, heap=hp, heap_free=free, heap_size=dsize)

            def name(o):
                return b[daddr + o:b.index(b"\0", daddr + o)].decode()

            def node(a):
                assert b[a:a + 4] == b"TREE" and b[a + 4] == 0
                lvl, n = struct.unpack_from("<BH", b, a + 5)
                assert struct.unpack_from("<QQ", b, a + 8) == (2**64 - 1, 2**64 - 1) or lvl >= 0
                keys, kids = [], []
                for i in range(n):
                    k, c = struct.unpack_from("<QQ", b, a + 24 + 16 * i)
                    keys.append(k)
                    kids.append(c)
                keys.append(struct.unpack_from("<Q", b, a + 24 + 16 * n)[0])
                names = []
                for i, c in enumerate(kids):
                    if lvl > 0:
                        names += node(c)
                        continue
                    assert b[c:c + 4] == b"SNOD" and b[c + 4] == 1
                    ns = struct.unpack_from("<H", b, c + 6)[0]
                    assert 1 <= ns <= 2 * self.leaf_k
                    here = []
                    for s in range(ns):
                        no, oh, cache = struct.unpack_from("<QQI", b, c + 8 + 40 * s)
                        here.append(name(no))
                        self._object(oh, path + "/" + name(no))
                        if cache == 1:  # cached B-tree / heap addresses must match the object's own message
                            got = self.objects[path + "/" + name(no)]
                            assert struct.unpack_from("<QQ", b, c + 8 + 40 * s + 24) == (got["btree"], got["heap"])
                    assert name(keys[i + 1]) == here[-1], "B-tree key = largest name of the child to its left"
                    names += here
                assert name(keys[0]) == "" or lvl > 0
                return names

            names = node(bt)
            assert names == sorted(names), "links are stored in strcmp order"
            self.objects[path or "/"]["links"] = names
            return
        space, dtype, layout = types[0x01][1], types[0x03][1], types[0x08][1]
        assert space[0] == 1
        rank = space[1]
        shape = list(struct.unpack_from("<%dQ" % rank, space, 8))
        assert layout[0] == 3
        kind = {1: "f32", 0: "i32", 3: "str"}[dtype[0] & 0xf]
        esize = struct.unpack_from("<I", dtype, 4)[0]
        data = b""
        if layout[1] == 1:
            addr_, size = struct.unpack_from("<QQ", layout, 2)
            assert size == int(np.prod(shape, dtype=np.int64)) * esize
            data = b[addr_:addr_ + size]
            assert addr_ % 8 == 0 and addr_ + size <= self.eof
        self.objects[path] = dict(kind=kind, shape=shape, esize=esize, data=data, layout_class=layout[1],
                                  messages={t: (fl, body) for t, fl, body in msgs})


def _read(L, path, dataset):
    dims = (ctypes.c_int64 * 8)()
    nd = ctypes.c_int()
    n = L.cos_hdf5_read_dataset(path.encode(), dataset.encode(), dims, 8, ctypes.byref(nd), None, 0)
    if n < 0:
        return None, None
    out = np.empty(n, np.float32)
    assert L.cos_hdf5_read_dataset(path.encode(), dataset.encode(), dims, 8, ctypes.byref(nd), out.ctypes.data, n) == n
    return out, list(dims[:nd.value])


def test_reader_is_pinned_on_libhdf5_written_fixtures(cos):
    from caffeonspark_b200 import _lib
    L = _lib.lib()
    raw = open(os.path.join(FIX, "solver_data.h5"), "rb").read()
    # independent of any parser: the two contiguous datasets sit at these offsets (layout messages in a hex dump)
    data = np.frombuffer(raw[0x860:0x860 + 8 * 3 * 10 * 10 * 4], np.float32)
    targets = np.frombuffer(raw[0x2de0:0x2de0 + 8 * 4], np.float32)
    got, shape = _read(L, os.path.join(FIX, "solver_data.h5"), "/data")
    assert shape == [8, 3, 10, 10] and np.array_equal(got, data)
    got, shape = _read(L, os.path.join(FIX, "solver_data.h5"), "targets")
    assert shape == [8, 1] and np.array_equal(got, targets)
    assert hashlib.sha256(data.tobytes()).hexdigest()[:16] == hashlib.sha256(raw[0x860:0x860 + 9600]).hexdigest()[:16]
    assert np.isfinite(data).all() and abs(float(data.std()) - 1.0) < 0.1  # generate_sample_data.py: randn
    # the Python mini-parser agrees dataset by dataset on both fixtures
    for fx in ("solver_data.h5", "sample_data.h5"):
        mini = MiniH5(os.path.join(FIX, fx))
        for path, o in mini.objects.items():
            if o["kind"] != "f32":
                continue
            got, shape = _read(L, os.path.join(FIX, fx), path)
            assert shape == o["shape"] and got.tobytes() == o["data"], (fx, path)
    # chunked + gzip: refused, never guessed
    got, _ = _read(L, os.path.join(FIX, "sample_data_2_gzip.h5"), "/data")
    assert got is None and b"not supported" in L.cos_last_error()


def _write_model(L, path, arrays, names):
    ptrs = (ctypes.c_void_p * len(arrays))(*[a.ctypes.data for a in arrays])
    nd = (ctypes.c_int * len(arrays))(*[a.ndim for a in arrays])
    dims = [d for a in arrays for d in a.shape]
    return L.cos_caffemodel_write_h5(path.encode(), len(arrays), (ctypes.c_char_p * len(names))(*[n.encode() for n in names]),
                                     nd, (ctypes.c_int64 * len(dims))(*dims), ptrs)


def test_written_model_has_the_structure_libhdf5_writes(cos, tmp_path):
    """Net::ToHDF5 layout (net.cpp:867-917): /data/<layer>/<j>; parsed by the independent Python mini-parser."""
    from caffeonspark_b200 import _lib
    L = _lib.lib()
    rng = np.random.RandomState(0)
    names = ["conv1", "conv1", "conv2", "conv2", "ip1", "ip1", "ip2", "ip2", "scale"]
    arrays = [rng.randn(20, 1, 5, 5), rng.randn(20), rng.randn(50, 20, 5, 5), rng.randn(50), rng.randn(500, 800),
              rng.randn(500), rng.randn(10, 500), rng.randn(10), rng.randn(3)]
    arrays = [a.astype(np.float32) for a in arrays]
    path = str(tmp_path / "m.caffemodel.h5")
    assert _write_model(L, path, arrays, names), L.cos_last_error()
    mini = MiniH5(path)
    assert mini.eof == os.path.getsize(path) and (mini.leaf_k, mini.internal_k) == (4, 16)
    assert mini.objects["/"]["links"] == ["data"]
    assert mini.objects["/data"]["links"] == ["conv1", "conv2", "ip1", "ip2", "scale"]
    j = {}
    for n, a in zip(names, arrays):
        k = j.get(n, 0)
        j[n] = k + 1
        o = mini.objects[f"/data/{n}/{k}"]
        assert o["kind"] == "f32" and o["shape"] == list(a.shape) and o["data"] == a.tobytes()
    # our reader, through the snapshot-level entry point (format recognised by the signature)
    out = np.empty(400000, np.float32)
    assert L.cos_caffemodel_read(path.encode(), b"ip1", 0, out.ctypes.data, out.size) == 400000
    assert np.array_equal(out, arrays[4].ravel())
    assert L.cos_caffemodel_read(path.encode(), b"conv2", 1, out.ctypes.data, out.size) == 50
    assert L.cos_caffemodel_read(path.encode(), b"nope", 0, None, 0) == -1
    # message bytes identical to what libhdf5 wrote for a float32 dataset
    ref = MiniH5(os.path.join(FIX, "solver_data.h5")).objects["/data"]["messages"]
    mine = mini.objects["/data/conv1/0"]["messages"]
    for t in (0x0003, 0x0005):  # datatype, fill value (flags + body)
        assert mine[t] == ref[t], hex(t)
    assert mine[0x0001][1][:8] == ref[0x0001][1][:8]  # dataspace: version 1, rank 4, max dims present
    assert mine[0x0008][1][:2] == ref[0x0008][1][:2] and mine[0x0008][0] == ref[0x0008][0]  # layout v3 contiguous
    # same message types (libhdf5 pads its 256-byte header block with a NIL message, type 0)
    assert sorted(mine) == sorted(t for t in ref if t != 0) == [0x01, 0x03, 0x05, 0x08, 0x12]
    assert mini.root_cache[0] == 1  # root entry caches B-tree / heap like libhdf5's


def test_solverstate_h5_round_trip_and_many_links(cos, tmp_path):
    """SnapshotSolverStateToHDF5 (sgd_solver.cpp:279-301): /iter, /learned_net, /current_step, /history/<i>.  16 history
    blobs (CaffeNet) need more than one symbol table node; names sort as strings ("0","1","10",...,"2")."""
    from caffeonspark_b200 import _lib
    L = _lib.lib()
    rng = np.random.RandomState(3)
    hist = [rng.randn(*s).astype(np.float32) for s in [(96, 3, 11, 11), (96,)] * 8]
    ptrs = (ctypes.c_void_p * len(hist))(*[a.ctypes.data for a in hist])
    nd = (ctypes.c_int * len(hist))(*[a.ndim for a in hist])
    dims = [d for a in hist for d in a.shape]
    path = str(tmp_path / "s.solverstate.h5")
    learned = "/some/dir/caffenet_iter_4500.caffemodel.h5"
    assert L.cos_solverstate_write_h5(path.encode(), 4500, 2, learned.encode(), len(hist), nd,
                                      (ctypes.c_int64 * len(dims))(*dims), ptrs), L.cos_last_error()
    mini = MiniH5(path)
    assert mini.objects["/"]["links"] == ["current_step", "history", "iter", "learned_net"]
    assert mini.objects["/history"]["links"] == sorted(str(i) for i in range(16))
    assert mini.objects["/iter"]["kind"] == "i32" and mini.objects["/iter"]["shape"] == [1]
    assert struct.unpack("<i", mini.objects["/iter"]["data"])[0] == 4500
    assert struct.unpack("<i", mini.objects["/current_step"]["data"])[0] == 2
    s = mini.objects["/learned_net"]
    assert s["kind"] == "str" and s["shape"] == [] and s["data"] == learned.encode() + b"\0"
    for i, a in enumerate(hist):
        assert mini.objects[f"/history/{i}"]["data"] == a.tobytes()
    it, step = ctypes.c_int(), ctypes.c_int()
    buf = ctypes.create_string_buffer(256)
    assert L.cos_solverstate_read(path.encode(), ctypes.byref(it), ctypes.byref(step), buf, 256, -1, None, 0) == 16
    assert (it.value, step.value, buf.value.decode()) == (4500, 2, learned)
    out = np.empty(hist[10].size, np.float32)
    assert L.cos_solverstate_read(path.encode(), None, None, None, 0, 10, out.ctypes.data, out.size) == hist[10].size
    assert np.array_equal(out, hist[10].ravel())  # numeric order restored: blob 10 is not the third name
    # swapped roles are rejected
    assert L.cos_caffemodel_read(path.encode(), b"conv1", 0, None, 0) == -1 and b"'data' group" in L.cos_last_error()


def test_truncated_and_foreign_hdf5_is_rejected(cos, tmp_path):
    from caffeonspark_b200 import _lib
    L = _lib.lib()
    a = [np.arange(24, dtype=np.float32).reshape(2, 3, 4)]
    path = str(tmp_path / "t.caffemodel.h5")
    assert _write_model(L, path, a, ["ip"])
    raw = open(path, "rb").read()
    for cut in (100, 300, 700, len(raw) - 8):
        p = tmp_path / f"cut{cut}.h5"
        p.write_bytes(raw[:cut])
        assert L.cos_caffemodel_read(str(p).encode(), b"ip", 0, None, 0) == -1
    bad = bytearray(raw)
    bad[8] = 2  # superblock version 2: new-style file
    (tmp_path / "v2.h5").write_bytes(bytes(bad))
    assert L.cos_caffemodel_read(str(tmp_path / "v2.h5").encode(), b"ip", 0, None, 0) == -1
    assert b"superblock" in L.cos_last_error()
    # a group with more than 256 links would need a two-level B-tree: refused at write time, not corrupted
    many = [np.zeros(1, np.float32)] * 300
    assert _write_model(L, str(tmp_path / "many.h5"), many, [f"l{i}" for i in range(300)]) == 0
    assert b"256 links" in L.cos_last_error()


def test_reader_never_crashes_on_mutated_files(cos, tmp_path):
    """Bounds checks: random byte mutations / truncations of a valid file must yield an error or a (different) parse,
    never a crash, a hang or an over-read (the reader slurps the file and checks every offset against its size)."""
    from caffeonspark_b200 import _lib
    L = _lib.lib()
    rng = np.random.RandomState(7)
    arrays = [rng.randn(4, 3).astype(np.float32), rng.randn(4).astype(np.float32), rng.randn(5).astype(np.float32)]
    path = str(tmp_path / "seed.caffemodel.h5")
    assert _write_model(L, path, arrays, ["ip1", "ip1", "ip2"])
    raw = bytearray(open(path, "rb").read())
    meta_end = 4000  # object headers, B-trees, heaps and symbol nodes live in the first few KB
    p = tmp_path / "mut.h5"
    outcomes = set()
    for trial in range(400):
        m = bytearray(raw)
        for _ in range(int(rng.randint(1, 6))):
            pos = int(rng.randint(8, min(len(m), meta_end)))
            m[pos] = int(rng.randint(0, 256)) if rng.rand() < 0.7 else (0xff if rng.rand() < 0.5 else 0x00)
        if rng.rand() < 0.1:
            m = m[:int(rng.randint(8, len(m)))]
        p.write_bytes(bytes(m))
        n = L.cos_caffemodel_read(str(p).encode(), b"ip1", 0, None, 0)
        outcomes.add(n)
        it, step = ctypes.c_int(), ctypes.c_int()
        L.cos_solverstate_read(str(p).encode(), ctypes.byref(it), ctypes.byref(step), None, 0, -1, None, 0)
    assert -1 in outcomes and 12 in outcomes  # some mutations are fatal, some are harmless
