"""The Nesterov, AdaGrad, RMSProp and AdaDelta solvers, host side (no GPU): what the solver parser accepts and
rejects, the solver fields of cos_solver_desc, and the CPU oracles of their updates."""
import math

import numpy as np
import pytest

import solver_numpy
import solver_oracle

NET = 'net_param { layer { name: "d" type: "Input" top: "x" input_param { shape { dim: 2 dim: 3 } } } ' \
      'layer { name: "ip" type: "InnerProduct" bottom: "x" top: "y" inner_product_param { num_output: 4 } } }\n'

# hyper-parameters of the reference's example solvers (caffe-public/examples/mnist/)
EXAMPLES = {
    "SGD": 'base_lr: 0.01 momentum: 0.9 weight_decay: 0.0005 lr_policy: "inv" gamma: 0.0001 power: 0.75',
    "Nesterov": 'base_lr: 0.01 momentum: 0.95 weight_decay: 0.0005 lr_policy: "step" gamma: 0.1 stepsize: 10000 '
                'type: "Nesterov"',
    "AdaGrad": 'base_lr: 0.01 weight_decay: 0.0005 lr_policy: "fixed" type: "AdaGrad"',
    "RMSProp": 'base_lr: 0.01 momentum: 0.0 weight_decay: 0.0005 lr_policy: "inv" gamma: 0.0001 power: 0.75 '
               'type: "RMSProp" rms_decay: 0.98',
    "AdaDelta": 'base_lr: 1.0 momentum: 0.95 weight_decay: 0.0005 lr_policy: "fixed" type: "AdaDelta" delta: 1e-6',
}


def _solver(tmp_path, text):
    p = tmp_path / "solver.prototxt"
    p.write_text(text + "\n" + NET)
    return str(p)


@pytest.mark.parametrize("type", sorted(EXAMPLES))
def test_parser_accepts_each_solver(cos, tmp_path, type):
    d = cos.parse_solver(_solver(tmp_path, EXAMPLES[type]))
    assert d.type == type and d.counts == [12, 4]
    f = np.float32
    assert f(d.delta) == f(1e-6 if type == "AdaDelta" else 1e-8)  # caffe.proto default 1e-8
    assert f(d.rms_decay) == f(0.98 if type == "RMSProp" else 0.0)  # no default: 0
    assert f(d.momentum) == f({"Nesterov": 0.95, "AdaDelta": 0.95, "SGD": 0.9}.get(type, 0.0))


@pytest.mark.parametrize("enum,type", [("SGD", "SGD"), ("NESTEROV", "Nesterov"), ("ADAGRAD", "AdaGrad"),
                                       ("RMSPROP", "RMSProp"), ("ADADELTA", "AdaDelta")])
def test_deprecated_solver_type_enum(cos, tmp_path, enum, type):
    text = EXAMPLES[type].replace(f'type: "{type}"', "") + f" solver_type: {enum}"
    assert cos.parse_solver(_solver(tmp_path, text)).type == type


@pytest.mark.parametrize("text,msg", [
    ('base_lr: 0.1 type: "AdaGrad" momentum: 0.9', "Momentum cannot be used with AdaGrad."),
    ('base_lr: 0.1 type: "RMSProp" momentum: 0.9 rms_decay: 0.9', "Momentum cannot be used with RMSProp."),
    ('base_lr: 0.1 type: "RMSProp" rms_decay: 1.0', "rms_decay should lie between 0 and 1."),
    ('base_lr: 0.1 type: "RMSProp" rms_decay: -0.1', "rms_decay should lie between 0 and 1."),
    ('base_lr: 0.1 solver_type: ADAGRAD momentum: 0.5', "Momentum cannot be used with AdaGrad."),
])
def test_constructor_checks(cos, tmp_path, text, msg):
    with pytest.raises(cos.CosError, match=msg.replace(".", r"\.")):
        cos.parse_solver(_solver(tmp_path, text))


@pytest.mark.parametrize("text", ['type: "Adam"', "solver_type: ADAM", 'type: "Nadam"', 'type: "nesterov"'])
def test_other_types_still_rejected(cos, tmp_path, text):
    with pytest.raises(cos.CosError, match="only SGD"):
        cos.parse_solver(_solver(tmp_path, "base_lr: 0.1 " + text))


def test_allocate_desc_applies_the_same_checks(cos):
    # the checks run before any device is touched, so they fail the same way on a machine without a GPU
    for kw, msg in [(dict(type="Adam"), "only SGD"), (dict(type="AdaGrad", momentum=0.9), "AdaGrad"),
                    (dict(type="RMSProp", rms_decay=1.5), "rms_decay")]:
        with pytest.raises(cos.CosError, match=msg):
            cos.CaffeNet(cos.SolverDesc([8], **kw))


@pytest.mark.parametrize("type", sorted(EXAMPLES))
def test_desc_round_trips_through_parse_solver(cos, tmp_path, type):
    d = cos.parse_solver(_solver(tmp_path, EXAMPLES[type]))
    c, keep = d.to_c()
    assert c.type.decode() == type
    assert np.float32(c.delta) == np.float32(d.delta) and np.float32(c.rms_decay) == np.float32(d.rms_decay)
    s = cos.SolverDesc([1], type=type)
    assert (s.type, s.delta, s.rms_decay) == (type, 1e-8, 0.0)


HP = {
    "SGD": dict(momentum=0.9),
    "Nesterov": dict(momentum=0.95),
    "AdaGrad": dict(momentum=0.0, delta=1e-8),
    "RMSProp": dict(momentum=0.0, rms_decay=0.98, delta=1e-8),
    "AdaDelta": dict(momentum=0.95, delta=1e-6),
}


def _split(hp):
    hp = dict(hp)
    return hp.pop("momentum"), hp


@pytest.mark.parametrize("type", solver_oracle.SOLVERS)
@pytest.mark.parametrize("N", range(1, 9))
def test_c_oracle_equals_numpy_restatement(oracle, type, N):
    rng = np.random.default_rng(1000 * N + solver_oracle.SOLVERS.index(type))
    for l1 in (False, True):
        for bf16 in (False, True):
            nb = int(rng.integers(1, 7))
            counts = [int(x) for x in rng.integers(0, 700, nb)]
            counts[0] += 1
            lm = [float(x) for x in rng.choice([0.5, 1.0, 2.0], nb)]
            dm = [float(x) for x in rng.choice([0.0, 1.0], nb)]
            m, extra = _split(HP[type])
            reg = "L1" if l1 else "L2"
            kw = dict(lr_policy="inv", base_lr=0.01, gamma=0.0001, power=0.75, momentum=m, weight_decay=0.0005,
                      seed=N + 3, bf16=bf16, regularization_type=reg)
            sim = solver_oracle.Simulation(N, counts, lm, dm, type=type, **extra, **kw)
            d = [w.copy() for w in sim.data]
            h = [x.copy() for x in sim.hist]
            h2 = [x.copy() for x in sim.hist2] if sim.hist2 is not None else None
            for t in range(5):
                grads = [sim.gradient(r, t) for r in range(N)]
                rate = sim.step([g.copy() for g in grads])
                solver_numpy.step(d, [g.copy() for g in grads], h, h2, counts, lm, dm, rate, m, 0.0005,
                                  regularization_type=reg, type=type, **extra)
                for r in range(N):
                    what = f"{type} N={N} {reg} bf16={bf16} iter {t} rank {r}"
                    assert np.array_equal(d[r].view(np.uint32), sim.data[r].view(np.uint32)), what + " weights"
                    assert np.array_equal(h[r].view(np.uint32), sim.hist[r].view(np.uint32)), what + " history"
                    if h2 is not None:
                        assert np.array_equal(h2[r].view(np.uint32), sim.hist2[r].view(np.uint32)), what + " h2"


def test_sgd_matches_the_sgd_oracle(oracle):
    """type SGD of the solver oracle is the existing SGD oracle, bit for bit."""
    counts, lm, dm = [300, 7, 1000, 3], [1, 2, 1, 2], [1, 0, 1, 0]
    hp = dict(lr_policy="fixed", base_lr=0.01, momentum=0.9, weight_decay=0.0005, seed=2)
    a = oracle.Simulation(3, counts, lm, dm, **hp)
    b = solver_oracle.Simulation(3, counts, lm, dm, type="SGD", **hp)
    for _ in range(3):
        a.step()
        b.step()
    assert all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(a.data, b.data))
    assert all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(a.hist, b.hist))


def _closed_form(type, g, h, h2, lr, m, delta, rms_decay):
    """test_gradient_based_solver.cpp:296-334 (reference) in double: the update value of one element."""
    update = lr * g
    temp = m * h
    if type == "SGD":
        update += temp
    elif type == "Nesterov":
        update += temp
        update = (1 + m) * update - temp
    elif type == "AdaGrad":
        update /= math.sqrt(h + g * g) + delta
    elif type == "RMSProp":
        update /= math.sqrt(rms_decay * h + g * g * (1 - rms_decay)) + delta
    elif type == "AdaDelta":
        avg = m * h + (1 - m) * (g * g)
        update = g * math.sqrt((h2 + delta) / (avg + delta)) * lr
    return update


@pytest.mark.parametrize("type", solver_oracle.SOLVERS)
def test_one_step_matches_the_reference_closed_form(oracle, type):
    rng = np.random.default_rng(7)
    P = 4096
    w = rng.uniform(-1, 1, P).astype(np.float32)
    g = (rng.choice([-1, 1], P) * rng.uniform(0.05, 1.0, P)).astype(np.float32)  # bounded away from zero
    h = rng.uniform(0.01, 0.5, P).astype(np.float32)
    h2 = rng.uniform(0.01, 0.5, P).astype(np.float32)
    m, extra = _split(HP[type])
    delta, rms_decay = np.float32(extra.get("delta", 1e-8)), np.float32(extra.get("rms_decay", 0.0))
    lr = np.float32(0.01)
    d, hh, hh2, gg = w.copy(), h.copy(), h2.copy(), g.copy()
    solver_oracle.apply_update(0, P, d, gg, hh, hh2 if type == "AdaDelta" else None, [P], [1.0], [1.0], lr, m, 0.0,
                               type=type, **extra)
    want = np.array([_closed_form(type, float(g[i]), float(h[i]), float(h2[i]), float(lr),
                                  float(np.float32(m)), float(delta), float(rms_decay)) for i in range(P)])
    np.testing.assert_allclose(gg, want, rtol=1e-5, atol=0)  # the update value ComputeUpdateValue leaves in diff
    np.testing.assert_array_equal(d, w - gg)  # Blob::Update
