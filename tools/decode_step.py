"""Time the real decode step (CUDA graph, Groma-7B LLaMA, B=16, ctx ~1030) and its GEMM-only / attention-only subsets.
A/B of builds via env: GROMA_B200_LIB.
    python tools/decode_step.py [ctx]"""
import os, sys, math, torch
sys.path.insert(0, ".")
from groma_b200.config import PathConfig
from groma_b200.synth import make_state_dict
from groma_b200.engine import GromaEngine
from groma_b200 import ops as G

ctx = int(sys.argv[1]) if len(sys.argv) > 1 else 1030
B = 16
cfg = PathConfig(box_score_thres=0.0)
sd = make_state_dict(cfg, seed=0, perturb_norms=False, dtype=torch.bfloat16, device="cuda")
eng = GromaEngine(cfg, sd)
del sd
eng.alloc_kv(B, 1100)
eng.kv.normal_(0, 0.5)
d = eng._decode_buffers(B)

def reset():
    d["ids"].fill_(1234); d["pos"].fill_(ctx); d["kv_len"].fill_(ctx)

def graph_of(fn):
    g = torch.cuda.CUDAGraph(); st = torch.cuda.Stream(); st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        fn()
        with torch.cuda.graph(g, stream=st, capture_error_mode="thread_local"):
            fn()
    torch.cuda.current_stream().wait_stream(st)
    return g

def timeit(g, reps=20):
    reset()
    for _ in range(3): g.replay()
    ts = []
    for _ in range(reps):
        reset()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); g.replay(); e1.record(); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    ts.sort(); return ts[len(ts) // 2]

reset()
g_step = graph_of(lambda: eng.decode_step(B))
ms = timeit(g_step)
Hd, I, V, L = cfg.llm_hidden, cfg.llm_inter, cfg.vocab + cfg.num_new_token, cfg.llm_layers
wbytes = L * (4 * Hd * Hd + 3 * Hd * I) * 2 + V * Hd * 2
kvbytes = L * 2 * B * ctx * Hd * 2
tag = " ".join(f"{k[6:]}={v}" for k, v in os.environ.items() if k.startswith("GROMA_"))
print(f"[{tag}] decode step: {ms:.3f} ms  ({(wbytes + kvbytes) / ms / 1e6:.0f} GB/s over weights {wbytes/1e9:.2f} GB + KV {kvbytes/1e9:.2f} GB)", flush=True)

sp = eng._decode_splits()
def one(wn, s, src):
    W = eng.w[wn]
    ws = d["ws"][: s * W.shape[0] * B].view(s, B, W.shape[0])
    G.gemm_swap_ab(d[src], W, ws, split_k=s, pdl=eng.use_pdl, transposed=True)
def gemms():
    for i in range(L):
        for wn, s, src in ((f"llm.{i}.qkv.w", sp["qkv"], "y"), (f"llm.{i}.o.w", sp["o"], "q"), (f"llm.{i}.gu.w", sp["gu"], "y"), (f"llm.{i}.down.w", sp["down"], "gu")):
            one(wn, s, src)
    one("head.w", sp["head"], "y")
ms_g = timeit(graph_of(gemms))
print(f"[{tag}]   splits {sp}", flush=True)
print(f"[{tag}]   GEMM-only graph: {ms_g:.3f} ms  {wbytes / ms_g / 1e6:.0f} GB/s", flush=True)
def attns():
    for i in range(L):
        G.decode_attention(d["q"], eng.kv[i, 0], eng.kv[i, 1], d["kv_len"], 1.0 / math.sqrt(128), d["a"], pdl=eng.use_pdl)
ms_a = timeit(graph_of(attns))
print(f"[{tag}]   attention-only graph: {ms_a:.3f} ms  {kvbytes / ms_a / 1e6:.0f} GB/s", flush=True)
