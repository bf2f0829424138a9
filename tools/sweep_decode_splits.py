"""Empirical split-K choice for the five swap-AB decode GEMM shapes (B=16): in-graph time of 24 back-to-back launches (PDL, weights
rotating over copies larger than L2) per split factor.   python tools/sweep_decode_splits.py"""
import sys, torch
sys.path.insert(0, ".")
from groma_b200 import ops as G

def timeit(fn, iters=20, warm=3):
    for _ in range(warm): fn()
    ts = []
    for _ in range(iters):
        s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
        s.record(); fn(); e.record(); torch.cuda.synchronize(); ts.append(s.elapsed_time(e))
    ts.sort(); return ts[len(ts) // 2] * 1000

B = 16
st = torch.cuda.Stream()
shapes = dict(qkv=(12288, 4096), o=(4096, 4096), gu=(22016, 4096), down=(4096, 11008), head=(32114, 4096))
only = sys.argv[1:] or list(shapes)
for name in only:
    N, K = shapes[name]
    copies = max(2, int(300e6 // (N * K * 2)) + 1)
    wl = [torch.randn(N, K, device="cuda").bfloat16() for _ in range(copies)]
    x = torch.randn(B, K, device="cuda").bfloat16()
    res = []
    for S in (1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 14, 16):
        if S > (K + 63) // 64: continue
        ws = torch.empty(S, B, N, device="cuda")
        def one(i):
            G.gemm_swap_ab(x, wl[i % copies], ws, split_k=S, pdl=True, transposed=True)
        g = torch.cuda.CUDAGraph()
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            one(0)
            with torch.cuda.graph(g, stream=st):
                for i in range(24): one(i)
        torch.cuda.current_stream().wait_stream(st)
        us = timeit(g.replay) / 24
        res.append((us, S))
        print(f"{name:5s} N={N} K={K} S={S:2d}: {us:6.2f} us  {N * K * 2 / us / 1e3:5.0f} GB/s", flush=True)
    best = min(res)
    print(f"{name:5s} best split {best[1]} at {best[0]:.2f} us = {N * K * 2 / best[0] / 1e3:.0f} GB/s", flush=True)
    del wl
    torch.cuda.empty_cache()
