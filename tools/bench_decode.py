"""Micro-benchmarks of the decode-step kernels at Groma-7B sizes (B=16, ctx~1000). CUDA events, rotating buffers."""
import sys, math, torch
sys.path.insert(0, ".")
from groma_b200 import ops as G
flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
def timeit(fn, iters=20, warm=3, do_flush=True):
    for _ in range(warm): fn()
    ts = []
    for _ in range(iters):
        if do_flush: flush.zero_()
        s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
        s.record(); fn(); e.record(); torch.cuda.synchronize(); ts.append(s.elapsed_time(e))
    ts.sort(); return ts[len(ts) // 2] * 1000
B, H, D, cap = 16, 32, 128, 1100
q = torch.randn(B, H * D, device="cuda").bfloat16(); kc = torch.randn(B, H, cap, D, device="cuda").bfloat16(); vc = torch.randn(B, H, cap, D, device="cuda").bfloat16()
out = torch.empty(B, H * D, device="cuda", dtype=torch.bfloat16)
for n in (966, 1030, 1093):
    kvl = torch.full((B,), n, dtype=torch.int32, device="cuda")
    us = timeit(lambda: G.decode_attention(q, kc, vc, kvl, 0.088, out))
    print(f"decode_attention ctx={n}: {us:.1f} us  {2*B*H*n*D*2/us/1e3:.0f} GB/s", flush=True)
Hd, I = 4096, 11008
x = torch.randn(B, Hd, device="cuda").bfloat16(); w = torch.ones(Hd, device="cuda"); y = torch.empty_like(x)
print(f"rmsnorm: {timeit(lambda: G.rmsnorm(x, w, 1e-5, out=y)):.1f} us")
for (N, S, act) in [(3 * Hd, 3, 0), (Hd, 13, 0), (2 * I, 6, 3), (Hd, 9, 0)]:
    ws = torch.randn(S, N, B, device="cuda"); o = torch.empty(B, N // 2 if act == 3 else N, device="cuda", dtype=torch.bfloat16)
    print(f"splitk_reduce N={N} S={S} act={act}: {timeit(lambda: G.splitk_reduce(ws, o, act=act, bias_along_m=True, ld_m=1, ld_n=o.shape[1])):.1f} us")
qkv = torch.randn(B, 3 * Hd, device="cuda").bfloat16(); qo = torch.empty(B, Hd, device="cuda", dtype=torch.bfloat16)
cos = torch.randn(4096, 64, device="cuda"); pos = torch.tensor([1000], dtype=torch.int32, device="cuda")
print(f"rope_kv: {timeit(lambda: G.rope_kv(qkv, qo, kc, vc, cos, cos, B, 1, H, D, 0, pos_ptr=pos)):.1f} us")
# back-to-back launch cost: 200 dependent tiny kernels in a CUDA graph
g = torch.cuda.CUDAGraph()
s = torch.cuda.Stream(); s.wait_stream(torch.cuda.current_stream())
with torch.cuda.stream(s):
    G.rmsnorm(x, w, 1e-5, out=y)
    with torch.cuda.graph(g, stream=s):
        for _ in range(200): G.rmsnorm(x, w, 1e-5, out=y)
torch.cuda.current_stream().wait_stream(s)
print(f"graph of 200 chained rmsnorm: {timeit(lambda: g.replay(), do_flush=False)/200:.2f} us per launch")
wq = [torch.randn(3 * Hd, Hd, device="cuda").bfloat16() for _ in range(8)]
ws = torch.empty(3, 3 * Hd, B, device="cuda")
g2 = torch.cuda.CUDAGraph()
with torch.cuda.stream(s):
    G.gemm_swap_ab(x, wq[0], ws, split_k=3)
    with torch.cuda.graph(g2, stream=s):
        for i in range(64): G.gemm_swap_ab(x, wq[i % 8], ws, split_k=3)
torch.cuda.current_stream().wait_stream(s)
us = timeit(lambda: g2.replay(), do_flush=False) / 64
print(f"graph of 64 chained qkv swap-AB GEMMs (100 MB each): {us:.1f} us per launch = {3*Hd*Hd*2/us/1e3:.0f} GB/s")

# ---- launch variants of the decode GEMM inside a realistic chain (rmsnorm -> GEMM -> reduce), CUDA graph
big = torch.randn(1 << 28, device="cuda")
print(f"torch.sum over 1 GiB fp32 (read-only stream): {big.numel()*4/timeit(lambda: big.sum(), iters=5)/1e3:.0f} GB/s")
del big
def chain(pdl, N, K, S, n=48):
    wl = [torch.randn(N, K, device="cuda").bfloat16() for _ in range(8)]
    xx = torch.randn(B, K, device="cuda").bfloat16(); yy = torch.empty_like(xx); wn = torch.ones(K, device="cuda")
    wsb = torch.empty(S, N, B, device="cuda"); oo = torch.empty(B, N, device="cuda", dtype=torch.bfloat16)
    def body(i):
        G.rmsnorm(xx, wn, 1e-5, out=yy)
        G.gemm_swap_ab(yy, wl[i % 8], wsb, split_k=S, pdl=pdl)
        G.splitk_reduce(wsb, oo, bias_along_m=True, ld_m=1, ld_n=N)
    g = torch.cuda.CUDAGraph()
    st = torch.cuda.Stream(); st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        body(0)
        with torch.cuda.graph(g, stream=st):
            for i in range(n): body(i)
    torch.cuda.current_stream().wait_stream(st)
    us = timeit(lambda: g.replay(), do_flush=False) / n
    ref = (yy.float() @ wl[(n - 1) % 8].float().t())
    err = ((oo.float() - ref).abs().max() / ref.abs().max()).item()
    print(f"chain N={N} K={K} S={S} pdl={int(pdl)}: {us:.1f} us per (norm+gemm+reduce)  weights {N*K*2/us/1e3:.0f} GB/s  err {err:.1e}", flush=True)
for (N, K, S) in [(12288, 4096, 3), (22016, 4096, 6), (4096, 11008, 9), (4096, 4096, 13)]:
    for pdl in (False, True):
        chain(pdl, N, K, S)
