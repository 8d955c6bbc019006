"""Microbenchmark of the F4C GEMM epilogue variants at the bench's row count (d3d_op_linear_bench act codes):
proj without / with the in-place residual, fc1 with its GELU epilogue, fc2 with its residual.

    python tools/gemm_epi_bench.py [M]
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from diff3dhpe_b200 import _lib  # noqa: E402
from diff3dhpe_b200.engine import Engine  # noqa: E402

M = int(sys.argv[1]) if len(sys.argv) > 1 else 2115072
eng = Engine(27, max_clips=1)
print(f"M={M} lib={_lib.LIB_PATH} EW_GELU={os.environ.get('D3D_GEMM_EW_GELU', '16')}")
for label, N, K, act in (("qkv  fp32 out", 1536, 512, 0), ("proj no residual", 512, 512, 0), ("proj + residual", 512, 512, 2),
                         ("fc1 gelu", 1024, 512, 1), ("fc2 no residual", 512, 1024, 0), ("fc2 + residual", 512, 1024, 2)):
    ms = eng.op_linear_bench(M, N, K, act, _lib.GEMM_TC_F4C, iters=5)
    print(f"{label:26s} N={N:4d} K={K:4d}: {ms:7.3f} ms  {2.0 * M * N * K / ms / 1e9:7.1f} TF/s algorithmic", flush=True)
