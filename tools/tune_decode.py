"""A/B of the decode swap-AB GEMM across builds on the B200: run as  [GROMA_B200_LIB=...] python tools/tune_decode.py"""
import os, sys, torch
sys.path.insert(0, ".")
from groma_b200 import ops as G
def timeit(fn, iters=30, warm=5):
    for _ in range(warm): fn()
    ts = []
    for _ in range(iters):
        s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
        s.record(); fn(); e.record(); torch.cuda.synchronize(); ts.append(s.elapsed_time(e))
    ts.sort(); return ts[len(ts) // 2] * 1000
B = 16
st = torch.cuda.Stream(); st.wait_stream(torch.cuda.current_stream())
Hd = 4096
for (N, K, S) in [(12288, 4096, 3), (22016, 4096, 6), (4096, 11008, 9)]:
    wl = [torch.randn(N, K, device="cuda").bfloat16() for _ in range(6)]
    x = torch.randn(B, K, device="cuda").bfloat16(); ws = torch.empty(S, B, N, device="cuda")
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.stream(st):
        G.gemm_swap_ab(x, wl[0], ws, split_k=S, transposed=True)
        with torch.cuda.graph(g2, stream=st):
            for i in range(24): G.gemm_swap_ab(x, wl[i % 6], ws, split_k=S, transposed=True)
    torch.cuda.current_stream().wait_stream(st)
    us = timeit(lambda: g2.replay()) / 24
    print(f"[lib={os.path.basename(os.environ.get('GROMA_B200_LIB','default'))}] swapAB N={N} K={K} S={S}: {us:.1f} us {N*K*2/us/1e3:.0f} GB/s", flush=True)
