"""Generates tests/golden/ref_kernel_vectors.npz and tests/golden/ref_kernel_checks.json by RUNNING the
reference's own C++ kernels (elasticdl/go/pkg/kernel/capi/kernel_api.cc of the reference tree, compiled unmodified
as oracle/_ref -- see oracle/Makefile `ref` and oracle/eigen_shim) on seeded inputs.  Needs the reference tree
(oracle/Makefile REF_CAPI):  python tests/golden/gen_kernel_vectors.py

Cases: SGD, Momentum, Nesterov, Adam and AMSGrad at steps 1 / 5 / 1000 / 100000 (the bias correction is
evaluated in double and narrowed, kernel_api.cc:67), Adagrad; sizes 1, 7 (ragged), 10 (kernel_test.go's
size), 515; three successive applications each so slot state feeds back.  Inputs include negatives,
zeros and tiny / large magnitudes.

ref_kernel_checks.json holds what the reference kernels returned for the inputs of tests/test_oracle_vs_ref.py,
so that those comparisons run without the reference tree:
* `live`: per seed (live_inputs) and case, the SHA-256 of every output array's fp32 bit patterns plus the bits at
  16 seeded positions (the full arrays would be ~2.7 MB);
* `kernel_test_go`: SGD and Adam on the inputs of kernel_test.go:25-47 / :69-107, every output bit pattern;
* `sparse_adam`: the four tables after sparse_adam_tables() with the reference's Adam applied per row.
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_kernels as R  # noqa: E402

F = np.float32


def inputs(rng, n):
    g = (rng.standard_normal(n) * 10.0 ** rng.integers(-4, 2, n)).astype(F)
    p = rng.standard_normal(n).astype(F)
    if n > 3:
        g[1] = 0.0
        p[2] = 0.0
        g[3] = F(1e-20)
    return g, p


def cases():
    """(name, kind, hyper-parameters, n) -- shared with the tests through the npz itself."""
    out = []
    for n in (1, 7, 10, 515):
        out.append(("sgd_n%d" % n, "sgd", dict(lr=0.1), n))
        out.append(("momentum_n%d" % n, "momentum", dict(mu=0.9, nesterov=0, lr=0.05), n))
        out.append(("nesterov_n%d" % n, "momentum", dict(mu=0.9, nesterov=1, lr=0.05), n))
        for step in (1, 5, 1000, 100000):
            out.append(("adam_s%d_n%d" % (step, n), "adam",
                        dict(lr=0.1 if step == 5 else 0.001, step=step, beta1=0.9, beta2=0.999, eps=1e-8, ams=0), n))
            out.append(("amsgrad_s%d_n%d" % (step, n), "adam",
                        dict(lr=0.001, step=step, beta1=0.9, beta2=0.999, eps=1e-8, ams=1), n))
        out.append(("adagrad_n%d" % n, "adagrad", dict(lr=0.05, eps=1e-7), n))
    return out


def run_ref(kind, hp, g3, p, s0, s1, s2):
    """Three applications in place with the reference kernels; gradient k of g3 in round k."""
    for k in range(3):
        g = np.ascontiguousarray(g3[k])
        if kind == "sgd":
            R.sgd(g, p, hp["lr"])
        elif kind == "momentum":
            R.momentum(g, p, s0, hp["mu"], hp["nesterov"], hp["lr"])
        elif kind == "adam":
            R.adam(g, p, s0, s1, hp["lr"], hp["step"] + k, hp["beta1"], hp["beta2"], hp["eps"],
                   s2 if hp["ams"] else None)
        elif kind == "adagrad":
            R.adagrad(g, p, s0, hp["lr"], hp["eps"])


LIVE_SEEDS = range(6)


def live_inputs(seed):
    """Fresh random inputs of one seed: a size in [1, 3000) that exercises the SSE body and the scalar tail, and
    one case of each kind / step.  Returns (n, [(name, kind, hp, g3, [p, s0, s1, s2])])."""
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 3000))
    out = []
    for name, kind, hp, _ in cases()[:13]:
        g3 = np.stack([inputs(rng, n)[0] for _ in range(3)])
        base = [rng.standard_normal(n).astype(F)] + [np.abs(rng.standard_normal(n)).astype(F) for _ in range(3)]
        out.append((name, kind, hp, g3, base))
    return n, out


def bits(a):
    return np.ascontiguousarray(a, dtype=F).view(np.uint32)


def digest(a):
    """SHA-256 of an fp32 array's little-endian bit patterns."""
    return hashlib.sha256(bits(a).astype("<u4").tobytes()).hexdigest()


def sample_positions(seed, n):
    return np.sort(np.random.default_rng(1000 + seed).choice(n, min(n, 16), replace=False))


def kernel_test_go_inputs():
    """elasticdl/go/pkg/kernel/kernel_test.go:25-47 (SGD: g, p) and :69-107 (Adam step 5: g, p, m, v)."""
    g = np.arange(10, dtype=F) * F(0.5) + F(0.25)
    p = np.arange(10, dtype=F) * F(-0.3) + F(1.0)
    rng = np.random.default_rng(3)
    return (g, p), tuple(rng.random(10).astype(F) for _ in range(4))


def sparse_adam_tables(dim, ref_adam=None):
    """The oracle's sparse Adam (oracle_sparse_adam: one Adam call per gradient row, duplicates applied in order) on
    400 rows with many duplicate ids, steps 1, 2 and 7, AMSGrad slot included.  ref_adam: a C Adam with the
    kernel_api.h signature applied per row instead of the restated one (the reference's, from oracle/_ref).
    Returns [params, m, v, max_square] rows 0..49."""
    import ctypes

    from oracle import ps_oracle as O

    rng = np.random.default_rng(dim)
    ids = rng.integers(0, 50, 400).astype(np.int64)
    grads = (rng.standard_normal((400, dim)) * 0.1).astype(F)
    O.lib.oracle_set_ref_adam(ctypes.cast(ref_adam, ctypes.c_void_p) if ref_adam is not None else None)
    try:
        tabs = [O.OracleTable(dim, "uniform", seed=3)] + [O.OracleTable(dim, "zero") for _ in range(3)]
        for step in (1, 2, 7):
            O.lib.oracle_sparse_adam(tabs[0]._h, tabs[1]._h, tabs[2]._h, tabs[3]._h, O._i64(ids), O._f32(grads),
                                     ids.size, 0.01, step, 0.9, 0.999, 1e-7)
        return [t.get(np.arange(50)) for t in tabs]
    finally:
        O.lib.oracle_set_ref_adam(None)


def main_checks():
    """tests/golden/ref_kernel_checks.json (see the module docstring)."""
    assert R.lib() is not None, "oracle/_ref not built (needs the reference tree)"
    live = {}
    for seed in LIVE_SEEDS:
        n, items = live_inputs(seed)
        pos = sample_positions(seed, n)
        per_case = {}
        for name, kind, hp, g3, base in items:
            a = [x.copy() for x in base]
            run_ref(kind, hp, g3, *a)
            per_case[name] = {k: {"sha256": digest(x), "sample": bits(x)[pos].tolist()}
                              for k, x in zip(("p", "s0", "s1", "s2"), a)}
        live[str(seed)] = {"n": n, "positions": pos.tolist(), "cases": per_case}
    (g, p), (g2, p0, m0, v0) = kernel_test_go_inputs()
    R.sgd(g, p, 0.1)
    p2, m2, v2 = p0.copy(), m0.copy(), v0.copy()
    R.adam(g2, p2, m2, v2, 0.1, 5, 0.9, 0.999, 1e-8)
    ktg = {"sgd_p": bits(p).tolist(), "adam_p": bits(p2).tolist(), "adam_m": bits(m2).tolist(),
           "adam_v": bits(v2).tolist()}
    sparse = {str(dim): [bits(t).reshape(-1).tolist() for t in sparse_adam_tables(dim, R.lib().Adam)] for dim in (1, 8)}
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_kernel_checks.json")
    with open(path, "w") as f:
        json.dump({"live": live, "kernel_test_go": ktg, "sparse_adam": sparse}, f, separators=(",", ":"))
        f.write("\n")
    print("wrote", path, os.path.getsize(path), "bytes")


def main():
    assert R.lib() is not None, "oracle/_ref not built (needs the reference tree)"
    rng = np.random.default_rng(20260921)
    out = {}
    names = []
    for name, kind, hp, n in cases():
        g3 = np.stack([inputs(rng, n)[0] for _ in range(3)])
        _, p = inputs(rng, n)
        s0 = np.abs(rng.standard_normal(n)).astype(F) * F(0.1)
        s1 = np.abs(rng.standard_normal(n)).astype(F) * F(0.01)
        s2 = np.abs(rng.standard_normal(n)).astype(F) * F(0.01)
        if kind == "adagrad":
            s0[:] = 0  # Q4: the Go PS starts the accumulator at 0
        out[name + "/g"] = g3
        for k, a in (("p", p), ("s0", s0), ("s1", s1), ("s2", s2)):
            out[name + "/in_" + k] = a.copy()
        run_ref(kind, hp, g3, p, s0, s1, s2)
        for k, a in (("p", p), ("s0", s0), ("s1", s1), ("s2", s2)):
            out[name + "/out_" + k] = a
        out[name + "/hp"] = np.array([kind] + ["%s=%r" % kv for kv in sorted(hp.items())])
        names.append(name)
    out["names"] = np.array(names)
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_kernel_vectors.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, len(names), "cases", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
    main_checks()
