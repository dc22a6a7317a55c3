"""The oracle against the reference's OWN compiled kernels (oracle/_ref) and against the vectors they produced.

* tests/golden/ref_kernel_vectors.npz was written by RUNNING the reference's kernel_api.cc (compiled unmodified,
  oracle/Makefile `ref`) -- tests/golden/gen_kernel_vectors.py.  The C restatement (ps_oracle.c) and its numpy twin
  must reproduce every output bit for bit.
* tests/golden/ref_kernel_checks.json holds what the same kernels returned on the seeded inputs of the other tests
  here (same generator): digests and samples of the outputs on fresh random inputs, kernel_test.go's own vectors, and
  the tables of the CPU arm's row-by-row sparse Adam.  The oracle must reproduce them; where oracle/_ref itself is
  present the oracle is also compared with it live.
Bar: bit-exact (integer compare of the fp32 patterns).
"""
import json
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import gen_kernel_vectors as G  # noqa: E402
from oracle import ps_oracle as O  # noqa: E402
from oracle import ref_kernels as R  # noqa: E402

F = np.float32
VEC = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_kernel_vectors.npz"))


def bits(a):
    return np.ascontiguousarray(a, dtype=F).view(np.uint32)


def run_oracle_c(kind, hp, g3, p, s0, s1, s2):
    for k in range(3):
        g = np.ascontiguousarray(g3[k])
        if kind == "sgd":
            O.lib.oracle_sgd(O._f32(g), O._f32(p), hp["lr"], p.size)
        elif kind == "momentum":
            O.lib.oracle_momentum(O._f32(g), O._f32(p), O._f32(s0), hp["mu"], hp["nesterov"], hp["lr"], p.size)
        elif kind == "adam":
            O.lib.oracle_adam(O._f32(g), O._f32(p), O._f32(s0), O._f32(s1), hp["lr"], p.size, hp["step"] + k,
                              hp["beta1"], hp["beta2"], hp["eps"], O._f32(s2) if hp["ams"] else O._null_f32())
        elif kind == "adagrad":
            O.lib.oracle_adagrad(O._f32(g), O._f32(p), O._f32(s0), hp["lr"], p.size, hp["eps"])


def run_oracle_np(kind, hp, g3, p, s0, s1, s2):
    for k in range(3):
        g = g3[k]
        if kind == "sgd":
            O.np_sgd(g, p, hp["lr"])
        elif kind == "momentum":
            O.np_momentum(g, p, s0, hp["mu"], hp["nesterov"], hp["lr"])
        elif kind == "adam":
            O.np_adam(g, p, s0, s1, hp["lr"], hp["step"] + k, hp["beta1"], hp["beta2"], hp["eps"],
                      s2 if hp["ams"] else None)
        elif kind == "adagrad":
            O.np_adagrad(g, p, s0, hp["lr"], hp["eps"])


CASES = {name: (kind, hp, n) for name, kind, hp, n in G.cases()}


def test_fixture_lists_the_generator_cases():
    assert list(VEC["names"]) == [c[0] for c in G.cases()]


@pytest.mark.parametrize("runner", [run_oracle_c, run_oracle_np], ids=["c", "numpy"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_reproduces_reference_kernel_vectors(name, runner):
    kind, hp, n = CASES[name]
    st = {k: VEC[name + "/in_" + k].copy() for k in ("p", "s0", "s1", "s2")}
    runner(kind, hp, VEC[name + "/g"], st["p"], st["s0"], st["s1"], st["s2"])
    for k in ("p", "s0", "s1", "s2"):
        assert np.array_equal(bits(st[k]), bits(VEC[name + "/out_" + k])), (name, k)


CHECKS = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_kernel_checks.json")))


def from_bits(b):
    return np.asarray(b, dtype=np.uint32).view(F)


def test_checks_fixture_covers_the_generator_inputs():
    assert sorted(CHECKS["live"]) == sorted(str(s) for s in G.LIVE_SEEDS)
    for seed in G.LIVE_SEEDS:
        n, items = G.live_inputs(seed)
        assert CHECKS["live"][str(seed)]["n"] == n
        assert sorted(CHECKS["live"][str(seed)]["cases"]) == sorted(c[0] for c in items)


@pytest.mark.parametrize("seed", range(6))
def test_oracle_equals_ref_live(seed):
    """Fresh random inputs each seed, sizes that exercise the SSE body and the scalar tail: the oracle's outputs
    equal the reference kernels' (stored digest of every array, bits at seeded positions; and live where
    oracle/_ref is present)."""
    n, items = G.live_inputs(seed)
    want = CHECKS["live"][str(seed)]
    pos = np.asarray(want["positions"])
    assert want["n"] == n and np.array_equal(pos, G.sample_positions(seed, n))
    ref = R.lib() is not None
    for name, kind, hp, g3, base in items:
        b = [x.copy() for x in base]
        run_oracle_c(kind, hp, g3, *b)
        for k, y in zip(("p", "s0", "s1", "s2"), b):
            w = want["cases"][name][k]
            assert np.array_equal(bits(y)[pos], np.asarray(w["sample"], dtype=np.uint32)), (name, k, n)
            assert G.digest(y) == w["sha256"], (name, k, n)
        if ref:
            a = [x.copy() for x in base]
            G.run_ref(kind, hp, g3, *a)
            for x, y in zip(a, b):
                assert np.array_equal(bits(x), bits(y)), (name, n)


def test_ref_replays_kernel_test_go_vectors():
    """elasticdl/go/pkg/kernel/kernel_test.go:25-47 (SGD, exact) and :69-107 (Adam step 5, expected
    values written with the Go-side formula, compared there with tolerance 1e-4... we keep 1e-6): the reference
    kernels' outputs (stored; live where oracle/_ref is present) meet them, and the oracle reproduces those
    outputs bit for bit."""
    want = CHECKS["kernel_test_go"]
    runs = [("stored", {k: from_bits(v) for k, v in want.items()})]
    if R.lib() is not None:
        (g, p), (g2, p0, m0, v0) = G.kernel_test_go_inputs()
        R.sgd(g, p, 0.1)
        p2, m2, v2 = p0.copy(), m0.copy(), v0.copy()
        R.adam(g2, p2, m2, v2, 0.1, 5, 0.9, 0.999, 1e-8)
        runs.append(("live", {"sgd_p": p, "adam_p": p2, "adam_m": m2, "adam_v": v2}))
    for label, r in runs:
        (g, p), (g2, p0, m0, v0) = G.kernel_test_go_inputs()
        assert np.array_equal(bits(r["sgd_p"]), bits(p - F(0.1) * g)), label
        em = 0.9 * m0.astype(np.float64) + 0.1 * g2
        ev = 0.999 * v0.astype(np.float64) + 0.001 * g2.astype(np.float64) ** 2
        ep = p0 - 0.1 * np.sqrt(1 - 0.999 ** 5) / (1 - 0.9 ** 5) * em / (np.sqrt(ev) + 1e-8)
        assert np.allclose(r["adam_m"], em, rtol=1e-6) and np.allclose(r["adam_v"], ev, rtol=1e-6), label
        assert np.allclose(r["adam_p"], ep, rtol=1e-5, atol=1e-6), label
        for k in want:
            assert np.array_equal(bits(r[k]), np.asarray(want[k], dtype=np.uint32)), (label, k)
    (g, p), (g2, p0, m0, v0) = G.kernel_test_go_inputs()
    O.lib.oracle_sgd(O._f32(g), O._f32(p), 0.1, p.size)
    O.lib.oracle_adam(O._f32(g2), O._f32(p0), O._f32(m0), O._f32(v0), 0.1, p0.size, 5, 0.9, 0.999, 1e-8, O._null_f32())
    for k, x in (("sgd_p", p), ("adam_p", p0), ("adam_m", m0), ("adam_v", v0)):
        assert np.array_equal(bits(x), np.asarray(want[k], dtype=np.uint32)), k


@pytest.mark.parametrize("dim", [1, 8])
def test_sparse_adam_rows_through_the_reference_kernel(dim):
    """The CPU arm of bench.py updates table rows with the reference's own compiled Adam (one call per row, as
    kernel.go:119-138 does through cgo): with the restated Adam the tables end up bit-identical to those the
    reference's Adam produced (stored; live where oracle/_ref is present), duplicates applied sequentially,
    AMSGrad slot included."""
    got = G.sparse_adam_tables(dim)
    want = CHECKS["sparse_adam"][str(dim)]
    assert len(got) == len(want) == 4
    for a, w in zip(got, want):
        assert np.array_equal(bits(a).reshape(-1), np.asarray(w, dtype=np.uint32))
    if R.lib() is not None:
        for a, b in zip(G.sparse_adam_tables(dim, R.lib().Adam), got):
            assert np.array_equal(bits(a), bits(b))
