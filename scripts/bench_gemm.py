"""The prefill GEMM alone: the fast drain q3_prefill runs vs the bit-identical exact drain (q3_bench_gemm_q8)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from qwen3_rs_b200 import transformer as T
shapes = [("4B qkv", 2048, 6144, 2560), ("4B o", 2048, 2560, 4096), ("4B gate/up", 2048, 19456, 2560), ("4B down", 2048, 2560, 9728),
          ("8B qkv", 2048, 6144, 4096), ("8B gate/up", 2048, 24576, 4096), ("8B down", 2048, 4096, 12288)]
print("tcgen05 int8 GEMM alone, T x N x K, gs 64; TOPS = 2*T*N*K / time; % of the 4500 TOPS datasheet figure in brackets")
print(f"{'shape':12s} {'T':>5s} {'N':>6s} {'K':>6s} | {'fast drain':>22s} | {'exact drain':>22s}")
for name, t, n, k in shapes:
    row = []
    for mode in (0, 1):
        ms = T.bench_gemm_q8(t, n, k, 64, mode, 5)
        tops = 2.0 * t * n * k / ms / 1e9
        row.append(f"{ms * 1e3:8.1f} us {tops:6.0f} ({tops / 45:4.1f}%)")
    print(f"{name:12s} {t:5d} {n:6d} {k:6d} | " + " | ".join(row))
