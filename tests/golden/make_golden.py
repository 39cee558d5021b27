"""Generates the fixtures under tests/golden/ from a checkout of the reference
project (CaffeOnSpark with its caffe-public submodule), so that the tests
that compare with the reference run without it:

    python tests/golden/make_golden.py <reference checkout>

* ref_sync_cases.npz / .json: what the reference's own socket-sync code
  computes (oracle/_ref/ref_sync = socket.cpp + socket_sync_cpu.cpp +
  parallel_cpu.cpp of the reference compiled verbatim, see oracle/Makefile),
  run as N loopback processes.
* ref_sync_digests.json: SHA-256 digests of ref_sync's float32 outputs for
  the cases tests/test_oracle.py pins, including the full LeNet layout
  (too large to store element by element).
* hdf5/*.h5: libhdf5-written fixtures of caffe-public's test data.
* configs/: the reference's solver / net prototxt files.
* reference_interfaces.json: the field numbers of the caffe.proto messages
  the snapshot files use, and the native methods CaffeNet.java declares.
"""
import hashlib
import json
import os
import re
import shutil
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402

CASES = [
    # name, N, counts, lr_mult, decay_mult, iters, seed, bf16, hyper
    ("n2_ragged_inv", 2, [50, 7, 33, 5], [1, 2, 1, 2], [1, 1, 1, 0], 4, 11, False,
     dict(lr_policy="inv", base_lr=0.01, gamma=0.0001, power=0.75, momentum=0.9, weight_decay=0.0005)),
    ("n3_odd_fixed", 3, [101, 3, 1, 64], [1, 2, 1, 2], [1, 0, 1, 0], 3, 12, False,
     dict(lr_policy="fixed", base_lr=0.001, momentum=0.9, weight_decay=0.004)),
    ("n4_step", 4, [1023], [1], [1], 5, 13, False,
     dict(lr_policy="step", base_lr=0.01, gamma=0.1, stepsize=2, momentum=0.9, weight_decay=0.0005)),
    ("n8_tiny", 8, [5, 2], [1, 2], [1, 1], 3, 14, False,
     dict(lr_policy="fixed", base_lr=0.05, momentum=0.5, weight_decay=0.0)),
    ("n2_bf16", 2, [130, 9], [1, 2], [1, 1], 3, 15, True,
     dict(lr_policy="fixed", base_lr=0.001, momentum=0.9, weight_decay=0.004)),
    ("n4_lenet_head", 4, [500, 20, 2500, 50], [1, 2, 1, 2], [1, 1, 1, 1], 3, 16, False,
     dict(lr_policy="inv", base_lr=0.01, gamma=0.0001, power=0.75, momentum=0.9, weight_decay=0.0005)),
    ("n5_multistep", 5, [333, 7, 64], [1, 2, 1], [1, 0, 1], 5, 17, False,
     dict(lr_policy="multistep", base_lr=0.02, gamma=0.5, stepvalues=(2, 4), momentum=0.9, weight_decay=0.001)),
    ("n6_poly", 6, [100, 1, 1, 1, 250], [1, 2, 1, 2, 1], [1, 1, 0, 0, 1], 3, 18, False,
     dict(lr_policy="poly", base_lr=0.01, power=2.0, max_iter=10, momentum=0.5, weight_decay=0.0005)),
    ("n7_plain_sgd", 7, [97, 11], [1, 1], [0, 0], 3, 19, False,
     dict(lr_policy="exp", base_lr=0.05, gamma=0.9, momentum=0.0, weight_decay=0.0)),
    ("n3_bf16_sigmoid", 3, [64, 64, 3], [1, 2, 1], [1, 1, 1], 3, 20, True,
     dict(lr_policy="sigmoid", base_lr=0.01, gamma=-0.5, stepsize=2, momentum=0.9, weight_decay=0.004)),
]

LENET_HP = dict(lr_policy="inv", base_lr=0.01, gamma=0.0001, power=0.75, momentum=0.9, weight_decay=0.0005)
DIGEST_CASES = [
    # name, N, counts, lr_mult, decay_mult, iters, seed, hyper
    ("ragged_n2", 2, [257, 3, 1021], [1, 2, 1], [1, 0, 1], 3, 21, LENET_HP),
    ("ragged_n3", 3, [257, 3, 1021], [1, 2, 1], [1, 0, 1], 3, 21, LENET_HP),
    ("lenet_n2", 2, [500, 20, 25000, 50, 400000, 500, 5000, 10], [1, 2] * 4, [1, 1] * 4, 3, 1, LENET_HP),
]

HDF5_FIXTURES = ["solver_data.h5", "sample_data.h5", "sample_data_2_gzip.h5"]
CONFIGS = {  # directory under configs/ -> (directory in the reference checkout, files)
    "data": ("data", ["lenet_memory_solver.prototxt", "lenet_memory_train_test.prototxt",
                      "cifar10_quick_solver.prototxt", "cifar10_quick_train_test.prototxt",
                      "bvlc_reference_solver.prototxt", "bvlc_reference_net.prototxt",
                      "lenet_cos_solver.prototxt", "lenet_cos_train_test.prototxt",
                      "lenet_dataframe_solver.prototxt", "lenet_dataframe_train_test.prototxt",
                      "lrcn_solver.prototxt"]),  # refused at clip_gradients, before its net is read
    "test_resources": ("caffe-distri/src/test/resources", ["caffenet_solver.prototxt",
                                                           "caffenet_train_net.prototxt"]),
}
PROTO_MESSAGES = ["BlobShape", "BlobProto", "LayerParameter", "NetParameter", "SolverState"]


def digest(a):
    """SHA-256 of the little-endian float32 bytes: equal digests mean bit-identical arrays."""
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<f4").tobytes()).hexdigest()


def ref_sync_cases():
    out, meta = {}, {}
    for name, N, counts, lm, dm, iters, seed, bf16, hp in CASES:
        ow, oh, fin = O.run_ref_dump(N, counts, lm, dm, iters=iters, seed=seed, bf16=bf16, **hp)
        for r in range(1, N):
            assert np.array_equal(fin[0], fin[r]), "ranks disagree after the trailing on_start"
        for t in range(iters):
            for r in range(N):
                out[f"{name}/w/{t}/{r}"] = ow[t][r]
                out[f"{name}/h/{t}/{r}"] = oh[t][r]
        out[f"{name}/final"] = fin[0]
        meta[name] = dict(N=N, counts=counts, lr_mult=lm, decay_mult=dm, iters=iters, seed=seed, bf16=bf16, hyper=hp)
    np.savez_compressed(os.path.join(HERE, "ref_sync_cases.npz"), **out)
    with open(os.path.join(HERE, "ref_sync_cases.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    print("wrote", len(out), "arrays for", len(meta), "cases")


def ref_sync_digests():
    cases = {}
    for name, N, counts, lm, dm, iters, seed, hp in DIGEST_CASES:
        ow, oh, fin = O.run_ref_dump(N, counts, lm, dm, iters=iters, seed=seed, **hp)
        cases[name] = dict(N=N, counts=counts, lr_mult=lm, decay_mult=dm, iters=iters, seed=seed, hyper=hp,
                           w=[[digest(ow[t][r]) for r in range(N)] for t in range(iters)],
                           h=[[digest(oh[t][r]) for r in range(N)] for t in range(iters)],
                           final=[digest(f) for f in fin])
    with open(os.path.join(HERE, "ref_sync_digests.json"), "w") as f:
        json.dump(cases, f, indent=1, sort_keys=True)
    print("wrote digests for", len(cases), "cases")


def copy_fixtures(ref):
    os.makedirs(os.path.join(HERE, "hdf5"), exist_ok=True)
    for fx in HDF5_FIXTURES:
        shutil.copyfile(os.path.join(ref, "caffe-public/src/caffe/test/test_data", fx), os.path.join(HERE, "hdf5", fx))
    for sub, (src, files) in CONFIGS.items():
        os.makedirs(os.path.join(HERE, "configs", sub), exist_ok=True)
        for fn in files:
            shutil.copyfile(os.path.join(ref, src, fn), os.path.join(HERE, "configs", sub, fn))


def reference_interfaces(ref):
    proto = open(os.path.join(ref, "caffe-public/src/caffe/proto/caffe.proto")).read()
    fields = {}
    for msg in PROTO_MESSAGES:
        body = re.search(r"message %s \{(.*?)\n\}" % msg, proto, re.S).group(1)
        decl = re.findall(r"^\s*(?:optional|repeated|required)\s+[\w.]+\s+(\w+)\s*=\s*(\d+)", body, re.M)
        fields[msg] = {name: int(number) for name, number in decl}
    java = open(os.path.join(ref, "caffe-distri/src/main/java/com/yahoo/ml/jcaffe/CaffeNet.java")).read()
    natives = sorted(set(re.findall(r"native\s+[\w\[\]]+\s+(\w+)\s*\(", java)))
    with open(os.path.join(HERE, "reference_interfaces.json"), "w") as f:
        json.dump({"caffe_proto_fields": fields, "caffenet_java_natives": natives}, f, indent=1, sort_keys=True)


def main():
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    ref = os.path.abspath(sys.argv[1])
    os.environ["REF"] = ref  # oracle/Makefile compiles ref_sync from $(REF)
    O.build(with_ref=True)
    assert O.ref_available(), "oracle/_ref/ref_sync was not built from " + ref
    ref_sync_cases()
    ref_sync_digests()
    copy_fixtures(ref)
    reference_interfaces(ref)


if __name__ == "__main__":
    main()
