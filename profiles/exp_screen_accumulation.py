"""How the BF16 screening kernels accumulate: FP32 sums of exact BF16 x BF16 products on the tensor cores.

The screening bound (csrc/screen_bf16.cu, kScreenUp) needs the accumulation error of K non-negative products.
Two probes per implementation (0: mma.sync, 1: tcgen05.mma):
  directed  row r = 1 + n_r small terms d_r (ulp(1) = 2^-23): round-to-nearest, truncation or a wider
            internal sum give different results
  random    non-negative BF16-exact operands with a wide exponent spread, exact reference by integer scaling:
            signed error (C - ref) / (K 2^-24 ref), its extremes and the share of elements above / below ref
Usage:  python profiles/exp_screen_accumulation.py OUT.json
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import revs_admm_b200 as R  # noqa: E402


def bf16_exact(rng, shape, e_lo, e_hi):
    m = rng.integers(128, 256, size=shape).astype(np.float64) / 128.0
    return m * np.exp2(rng.integers(e_lo, e_hi + 1, size=shape))


def exact_product(A, B, e_min_a, e_min_b):
    Ai, Bi = A * 2.0 ** (7 - e_min_a), B * 2.0 ** (7 - e_min_b)      # integers
    assert Ai.max() * Bi.max() * A.shape[1] < 2.0 ** 53
    return (Ai @ Bi) * 2.0 ** (e_min_a + e_min_b - 14)


def directed(impl):
    # row: A[r, 0] = 1 plus n small terms d at k = 1..n (same k block) or k = 16..16+n-1 (next block); B = 1
    cases = [(d, n, k0) for d in (0.25, 0.5, 0.75, 1.0, 1.5) for n in (1, 3, 15) for k0 in (1, 16)]
    K, T = 64, 8
    A = np.zeros((len(cases), K))
    for r, (d, n, k0) in enumerate(cases):
        A[r, 0] = 1.0
        A[r, k0:k0 + n] = d * 2.0 ** -23
    C = R.screen_contract(A, np.ones((K, T)), impl=impl)
    out = []
    for r, (d, n, k0) in enumerate(cases):
        out.append(dict(term_ulps=d, terms=n, first_k=k0, exact_ulps=d * n, result_ulps=float((C[r, 0] - 1.0) / 2.0 ** -23)))
    return out


def random_runs(impl, rng):
    res = []
    for K in (16, 64, 1024, 16384):
        M, T = 256, 96
        A, B = bf16_exact(rng, (M, K), -12, -4), bf16_exact(rng, (K, T), -4, 4)
        A *= rng.random((M, K)) < 0.8
        C = R.screen_contract(A, B, impl=impl)
        ref = exact_product(A, B, -12, -4)
        e = (C - ref) / (K * 2.0 ** -24 * ref)
        res.append(dict(K=K, err_min=float(e.min()), err_max=float(e.max()), share_above=float((C > ref).mean()),
                        share_below=float((C < ref).mean())))
    return res


def main():
    rng = np.random.default_rng(7)
    out = {"device": R.device_count() and os.popen("nvidia-smi --query-gpu=name,power.limit --format=csv,noheader").read().strip()}
    for impl in (0, 1):
        out[f"impl{impl}"] = dict(directed=directed(impl), random=random_runs(impl, rng))
    js = json.dumps(out, indent=1)
    print(js)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(js + "\n")


if __name__ == "__main__":
    main()
