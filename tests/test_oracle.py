"""CPU tests of the ORACLE itself: pins oracle/sync_oracle.c against
 (1) golden vectors produced by the reference's own socket-sync code
     (tests/golden/make_golden.py, run against a reference checkout),
 (2) digests of the reference binary's outputs stored the same way, and the
     binary itself when oracle/_ref was built,
 (3) the analytic least-squares SGD update of the reference's
     test_gradient_based_solver.cpp:224-347 (tolerance of :349-397),
 (4) the invariants of SURVEY.md section 8c.
"""
import hashlib
import json
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _cases():
    with open(os.path.join(GOLD, "ref_sync_cases.json")) as f:
        return json.load(f)


def _digest(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<f4").tobytes()).hexdigest()


def _check_against_reference_digests(oracle, name):
    """The oracle reproduces, bit for bit, what the reference binary computed for case `name` of
    ref_sync_digests.json; when oracle/_ref was built, the binary is run again and must still agree."""
    with open(os.path.join(GOLD, "ref_sync_digests.json")) as f:
        m = json.load(f)[name]
    N, iters = m["N"], m["iters"]
    sim = oracle.Simulation(N, m["counts"], m["lr_mult"], m["decay_mult"], seed=m["seed"], **m["hyper"])
    for t in range(iters):
        sim.step()
        for r in range(N):
            w, h = sim.own(r)
            assert _digest(w) == m["w"][t][r], f"weights differ at iter {t} rank {r}"
            assert _digest(h) == m["h"][t][r], f"history differs at iter {t} rank {r}"
    assert m["final"] == [_digest(sim.consistent_weights())] * N
    if oracle.ref_available():
        ow, oh, fin = oracle.run_ref_dump(N, m["counts"], m["lr_mult"], m["decay_mult"], iters=iters, seed=m["seed"],
                                          **m["hyper"])
        assert [[_digest(x) for x in row] for row in ow] == m["w"] and [[_digest(x) for x in row] for row in oh] == m["h"]
        assert [_digest(f) for f in fin] == m["final"]
    return m


@pytest.mark.parametrize("name", sorted(_cases().keys()))
def test_oracle_matches_reference_golden_vectors(oracle, name):
    meta = _cases()[name]
    gold = np.load(os.path.join(GOLD, "ref_sync_cases.npz"))
    sim = oracle.Simulation(meta["N"], meta["counts"], meta["lr_mult"], meta["decay_mult"], seed=meta["seed"],
                            bf16=meta["bf16"], **meta["hyper"])
    for t in range(meta["iters"]):
        sim.step()
        for r in range(meta["N"]):
            w, h = sim.own(r)
            assert np.array_equal(w, gold[f"{name}/w/{t}/{r}"]), f"weights differ at iter {t} rank {r}"
            assert np.array_equal(h, gold[f"{name}/h/{t}/{r}"]), f"history differs at iter {t} rank {r}"
    assert np.array_equal(sim.consistent_weights(), gold[f"{name}/final"])


def test_oracle_matches_reference_binary_live(oracle):
    for name in ("ragged_n2", "ragged_n3"):
        _check_against_reference_digests(oracle, name)


def test_chunk_known_answers(oracle):
    # socket_sync_cpu.cpp:46-54: start = peer*P/N, until = (peer+1)*P/N (integer, multiply first)
    for P, N in [(431080, 2), (431080, 8), (145578, 4), (60965224, 8), (7, 3), (1, 2), (5, 8), (2 ** 31 + 5, 3)]:
        prev = 0
        for r in range(N):
            o, s = oracle.chunk(P, N, r)
            assert o == r * P // N and s == (r + 1) * P // N - r * P // N
            assert o == prev
            prev = o + s
        assert prev == P
    assert oracle.chunk(431080, 8, 3) == (161655, 53885)
    assert oracle.chunk(60965224, 8, 7) == (53344571, 7620653)


def test_total_size_rule(oracle):
    assert oracle.total_size([500, 20]) == 520
    assert oracle.total_size([]) == 1  # parallel.cpp:66-67: at least one element


def test_learning_rate_policies(oracle):
    lr = oracle.learning_rate
    assert lr("fixed", 0.001) == pytest.approx(0.001, rel=1e-7)
    # LeNet: inv, base 0.01, gamma 1e-4, power 0.75 (data/lenet_memory_solver.prototxt)
    for it in (0, 1, 100, 1999):
        want = 0.01 * (1 + 1e-4 * it) ** -0.75
        assert lr("inv", 0.01, 1e-4, 0.75, it=it) == pytest.approx(want, rel=2e-6)
    # CaffeNet: step, gamma 0.1, stepsize 100000
    assert lr("step", 0.01, 0.1, stepsize=100000, it=99999) == pytest.approx(0.01, rel=1e-6)
    assert lr("step", 0.01, 0.1, stepsize=100000, it=100000) == pytest.approx(0.001, rel=1e-6)
    st = oracle.LrState()
    got = [lr("multistep", 1.0, 0.5, stepvalues=(2, 4), it=i, state=st) for i in range(6)]
    assert got == pytest.approx([1, 1, 0.5, 0.5, 0.25, 0.25])
    assert lr("poly", 0.1, power=2.0, max_iter=10, it=5) == pytest.approx(0.1 * 0.25, rel=1e-6)
    assert lr("exp", 0.1, 0.9, it=3) == pytest.approx(0.1 * 0.9 ** 3, rel=1e-6)
    assert lr("sigmoid", 0.1, -0.5, stepsize=4, it=4) == pytest.approx(0.05, rel=1e-6)


def test_fill_generator_twins_agree(oracle):
    for n, seed, stream, amp in [(1000, 7, 3, 0.01), (17, 1, 0, 0.05), (4097, 99, 4096 * 3 + 2, 1.0)]:
        assert np.array_equal(oracle.fill(n, seed, stream, amp), oracle.fill_numpy(n, seed, stream, amp))


def test_single_rank_is_plain_sgd(oracle):
    # N == 1 degenerates to single-process SGD (no scale, no exchange)
    counts, lm, dm = [37, 5], [1, 2], [1, 0]
    sim = oracle.Simulation(1, counts, lm, dm, lr_policy="fixed", base_lr=0.1, momentum=0.9, weight_decay=0.01, seed=3)
    w = sim.data[0].astype(np.float64).copy()
    h = np.zeros_like(w)
    lr = np.repeat(np.array(lm) * np.float32(0.1), counts).astype(np.float64)
    ld = np.repeat(np.array(dm) * np.float32(0.01), counts).astype(np.float64)
    for t in range(4):
        g = sim.gradient(0, t).astype(np.float64)
        sim.step()
        h = 0.9 * h + lr * (g + ld * w)
        w = w - h
    assert np.allclose(sim.data[0], w, rtol=1e-5, atol=1e-7)


def test_all_ranks_equal_after_on_start(oracle):
    N, P = 5, 1003
    data = [oracle.fill(P, 50 + r, 0, 1.0) for r in range(N)]  # deliberately different per rank
    want = np.empty(P, np.float32)
    for r in range(N):
        o, s = oracle.chunk(P, N, r)
        want[o:o + s] = data[r][o:o + s]
    oracle.all_gather(data)
    for r in range(N):
        assert np.array_equal(data[r], want)


def test_reduce_order_is_the_references(oracle):
    # owner r adds peers r+1, r+2, ... in that order, each pre-scaled by fl(1/N)
    N, P = 3, 9
    rng = np.random.RandomState(0)
    diff = [(rng.randn(P) * 10 ** rng.uniform(-3, 3, P)).astype(np.float32) for _ in range(N)]
    inv = np.float32(1.0 / N)
    want = []
    for r in range(N):
        o, s = oracle.chunk(P, N, r)
        acc = inv * diff[r][o:o + s]
        for j in range(1, N):
            acc = (inv * diff[(r + j) % N][o:o + s]) + acc
        want.append(acc.astype(np.float32))
    d2 = [d.copy() for d in diff]
    for d in d2:
        oracle.scale(N, d)
    oracle.reduce_scatter(d2)
    for r in range(N):
        o, s = oracle.chunk(P, N, r)
        assert np.array_equal(d2[r][o:o + s], want[r])


@pytest.mark.parametrize("lr,wd,mom,iters", [(1.0, 0.0, 0.0, 1), (0.01, 0.5, 0.0, 1), (0.01, 0.0, 0.5, 4),
                                              (0.01, 0.5, 0.9, 4)])
def test_update_matches_analytic_least_squares(oracle, lr, wd, mom, iters):
    """test_gradient_based_solver.cpp:224-347 ComputeLeastSquaresUpdate with the
    constants of :574-636, checked to CheckLeastSquaresUpdate's tolerance
    max(1e-7, 1e-2 * min|.|) (:349-397)."""
    rng = np.random.RandomState(1701)
    n, D = 8, 3 * 10 * 10  # solver_data.h5: 8 x 3x10x10 data, 8 targets
    X = rng.randn(n, D)
    y = rng.randn(n)
    Xa = np.hstack([X, np.ones((n, 1))])
    theta = np.concatenate([rng.randn(D) * 0.01, [0.0]])  # weights + bias, float64 analytic track
    hist = np.zeros(D + 1)
    w32 = theta.astype(np.float32).copy()
    h32 = np.zeros(D + 1, np.float32)
    for _ in range(iters):
        # analytic: grad = X^T(X theta - y)/N + wd*theta ; update = lr*grad + momentum*history
        grad = Xa.T @ (Xa @ theta - y) / n + wd * theta
        upd = lr * grad + mom * hist
        hist = upd
        theta = theta - upd
        # oracle: same raw gradient (without decay) fed to the restated ApplyUpdate
        g32 = (Xa.T @ (Xa @ w32.astype(np.float64) - y) / n).astype(np.float32)
        oracle.apply_update(0, D + 1, w32, g32, h32, [D, 1], [1.0, 1.0], [1.0, 1.0], np.float32(lr),
                            np.float32(mom), np.float32(wd))
    tol = np.maximum(1e-7, 1e-2 * np.minimum(np.abs(theta), np.abs(w32)))
    assert np.all(np.abs(theta - w32) <= tol + 1e-6)


def test_bf16_rounding_is_rne(oracle):
    x = np.array([1.0, 1.00390625, 1.01171875, -3.14159, 65504.0, 1e-40, 0.0], np.float32)
    got = oracle.round_bf16(x)
    import torch
    want = torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()
    assert np.array_equal(got, want)


def test_baseline_config0_lenet_two_cpu_executors(oracle):
    """BASELINE.json configs[0]: LeNet (lenet_memory_solver.prototxt hyper-parameters, P = 431,080), 2 CPU
    executors, the reference's own socket sync (its outputs stored as digests, re-run when oracle/_ref exists)
    matched bit for bit by the C restatement.  This is the plumbing case that needs no GPU."""
    m = _check_against_reference_digests(oracle, "lenet_n2")
    assert m["N"] == 2 and m["counts"] == [500, 20, 25000, 50, 400000, 500, 5000, 10]
    assert m["hyper"] == dict(lr_policy="inv", base_lr=0.01, gamma=0.0001, power=0.75, momentum=0.9, weight_decay=0.0005)
    assert m["final"][0] == m["final"][1]
    assert sum(m["counts"]) == 431080 and oracle.chunk(431080, 2, 1) == (215540, 215540)


def test_c_oracle_agrees_with_independent_numpy_restatement(oracle):
    """Two restatements written separately (C scalar loops vs vectorised numpy) must agree bit for bit on
    random layouts, world sizes and hyper-parameters."""
    from oracle import numpy_oracle as NO
    rng = np.random.RandomState(2024)
    for trial in range(40):
        N = int(rng.randint(1, 9))
        nb = int(rng.randint(1, 6))
        counts = [int(c) for c in rng.randint(1, 200, nb)]
        lm = [float(x) for x in rng.choice([1.0, 2.0, 0.5], nb)]
        dm = [float(x) for x in rng.choice([1.0, 0.0, 0.25], nb)]
        P = sum(counts)
        rate, mom, wd = np.float32(rng.uniform(1e-4, 0.1)), np.float32(rng.choice([0.0, 0.5, 0.9])), \
            np.float32(rng.choice([0.0, 5e-4, 4e-3]))
        data = [(rng.randn(P) * 0.05).astype(np.float32) for _ in range(N)]
        hist = [(rng.randn(P) * 0.01).astype(np.float32) for _ in range(N)]
        grads = [(rng.randn(P) * 10 ** rng.uniform(-4, 0)).astype(np.float32) for _ in range(N)]
        reg = "L1" if trial % 3 == 2 else "L2"  # sgd_solver.cpp:161-168: g += local_decay * sign(w)
        if reg == "L1":
            data[0][: min(3, P)] = [0.0, -0.0, 1.0][: min(3, P)]  # sign(+-0) = 0
        want_d, want_h = NO.step(data, grads, hist, counts, lm, dm, rate, mom, wd, reg)
        d2 = [x.copy() for x in data]
        h2 = [x.copy() for x in hist]
        g2 = [x.copy() for x in grads]
        oracle.step(d2, g2, h2, counts, lm, dm, rate, mom, wd, reg)
        for r in range(N):
            assert np.array_equal(d2[r].view(np.uint32), want_d[r].view(np.uint32)), (trial, N, r)
            assert np.array_equal(h2[r].view(np.uint32), want_h[r].view(np.uint32)), (trial, N, r)


def test_l1_regularization_known_answers(oracle):
    """Regularize with regularization_type "L1" (sgd_solver.cpp:161-168): diff += local_decay * sign(data), then
    the usual momentum update.  Hand-computed on exactly representable numbers."""
    data = np.array([2.0, -4.0, 0.0, -0.0], np.float32)
    diff = np.array([1.0, 1.0, 1.0, 1.0], np.float32)
    hist = np.zeros(4, np.float32)
    # rate 0.5, momentum 0, weight_decay 0.25, lr_mult 1, decay_mult 2 -> local_decay 0.5
    oracle.apply_update(0, 4, data, diff, hist, [4], [1.0], [2.0], np.float32(0.5), np.float32(0.0), np.float32(0.25), "L1")
    assert hist.tolist() == [0.75, 0.25, 0.5, 0.5]          # lr * (g + 0.5*sign(w))
    assert data.tolist() == [1.25, -4.25, -0.5, -0.5]
    d2, g2, h2 = np.array([2.0, -4.0], np.float32), np.array([1.0, 1.0], np.float32), np.zeros(2, np.float32)
    oracle.apply_update(0, 2, d2, g2, h2, [2], [1.0], [2.0], np.float32(0.5), np.float32(0.0), np.float32(0.25))  # L2
    assert h2.tolist() == [1.0, -0.5] and d2.tolist() == [1.0, -3.5]
