"""Sustained (power-capped) time of the encoder GEMM shapes."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.argv = [sys.argv[0], "none"]
import power_probe as pp
M = int(os.environ.get("M", "29316"))
for (N, K, act) in [(3072, 1024, -2), (1024, 1024, -3), (4096, 1024, -2), (1024, 4096, -3)]:
    pp.gemm(M, N, K, 0, act, 2.0)
