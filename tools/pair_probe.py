"""The GEMM core on the denoiser's shapes.
Build with -DMSMD_GEMM_TRACE and set MSMD_GEMM_TRACE=1 for the per-role clock64 timeline of CTAs 0, 1, 77."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tools.gemm_bench as gb
M = 21312
for N, K, act in [(1536, 128, 0), (1536, 512, 0), (1536, 1024, 0), (512, 512, 0), (512, 2048, 0), (2048, 512, 1)]:
    gb.bench(M, N, K, act=act, cublas=False)
