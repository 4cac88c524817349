"""Times the decoder's GEMM shapes at M = 15 000 rows (1 000 queries x beam 15) through sealdec_debug_gemm, gemm_mode 5.

    python tools/gemm_shapes.py [--root DIR] [--iters N] [--reps R]

--root picks the checkout whose seal_b200/libsealb200.so is loaded (default: this one), so two builds can be compared
in one session.  Times are CUDA events over N back-to-back calls (each call also splits A into fp16 halves: ~61 MB
read, 61 MB written at K = 1024); the best of R repetitions is kept.  The operands fit in L2 except A of fc2.
Prints one JSON line per shape: us per call and the tensor rate 3 x 2MNK / time (3 fp16 passes).
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

SHAPES = [("qkv", 3072, 1024, False), ("o", 1024, 1024, False), ("cq", 1024, 1024, False), ("co", 1024, 1024, False),
          ("fc1_gelu", 4096, 1024, True), ("fc2", 1024, 4096, False), ("lm_head", 50265, 1024, False)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--rows", type=int, default=15000)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    from seal_b200._lib import lib, check
    M = args.rows
    rng = np.random.default_rng(0)
    for name, N, K, gelu in SHAPES:
        A = rng.standard_normal((M, K)).astype(np.float32)
        W = (rng.standard_normal((N, K)) * 0.05).astype(np.float32)
        b = rng.standard_normal(N).astype(np.float32)
        out = np.empty((M, N), dtype=np.float32)
        best = float("inf")
        for _ in range(args.reps):
            us = C.c_double(0)
            check(lib.sealdec_debug_gemm(5, M, N, K, A.ctypes.data, W.ctypes.data, b.ctypes.data, out.ctypes.data,
                                         int(gelu), args.iters, C.byref(us)))
            best = min(best, us.value)
        print(json.dumps({"root": os.path.basename(os.path.abspath(args.root)), "shape": name, "M": M, "N": N, "K": K,
                          "gelu": gelu, "us": round(best, 1), "tensor_pflops": round(3 * 2.0 * M * N * K / best / 1e9, 3)}),
              flush=True)


if __name__ == "__main__":
    main()
