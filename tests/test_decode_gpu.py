"""Decode-path kernels: single-query attention over the KV cache and the swap-AB GEMM + transposing reduce epilogues."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def G():
    from groma_b200 import ops
    return ops


def rnd(*shape, seed=0, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale


def test_decode_attention_matches_reference(G):
    B, H, D, cap = 5, 4, 128, 300
    q = rnd(B, H * D, seed=1).bfloat16()
    kc = rnd(B, H, cap, D, seed=2).bfloat16()
    vc = rnd(B, H, cap, D, seed=3).bfloat16()
    kv_len = torch.tensor([300, 1, 2, 33, 257], dtype=torch.int32)
    scale = 1.0 / math.sqrt(D)
    out = torch.empty(B, H * D, dtype=torch.bfloat16, device="cuda")
    G.decode_attention(q.cuda(), kc.cuda(), vc.cuda(), kv_len.cuda(), scale, out)
    for b in range(B):
        n = int(kv_len[b])
        s = torch.einsum("hd,hkd->hk", q[b].float().reshape(H, D), kc[b, :, :n].float()) * scale
        want = torch.einsum("hk,hkd->hd", torch.softmax(s, -1), vc[b, :, :n].float()).reshape(-1)
        err = (out[b].float().cpu() - want).abs().max() / want.abs().max()
        assert err < 1e-2, (b, err.item())
    # agrees with the tensor-core kernel used for prefill on the same cache
    a2 = G.attention(q.cuda().reshape(B, 1, H, D), kc.cuda(), vc.cuda(), causal=False, scale=scale, kv_len=kv_len.cuda())
    assert (a2.reshape(B, -1).float() - out.float()).abs().max() < 2e-2


def test_swap_ab_reduce_epilogues(G):
    B, K, N = 16, 512, 768
    x = rnd(B, K, seed=4).bfloat16(); w = rnd(N, K, seed=5, scale=0.05).bfloat16(); res = rnd(B, N, seed=6).bfloat16()
    ref = x.float() @ w.float().t()
    for split in (1, 3, 5):
        ws = torch.empty(split, N, B, dtype=torch.float32, device="cuda")
        G.gemm_swap_ab(x.cuda(), w.cuda(), ws, split_k=split)
        out = torch.empty(B, N, dtype=torch.bfloat16, device="cuda")
        G.splitk_reduce(ws, out, residual=res.cuda(), bias_along_m=True, ld_m=1, ld_n=N)
        want = ref + res.float()
        assert ((out.float().cpu() - want).abs().max() / want.abs().max()) < 6e-3
        # SwiGLU over interleaved (gate, up) weight rows -> [B, N/2]
        o2 = torch.empty(B, N // 2, dtype=torch.bfloat16, device="cuda")
        G.splitk_reduce(ws, o2, act=G.ACT_SWIGLU, bias_along_m=True, ld_m=1, ld_n=N // 2)
        want2 = F.silu(ref[:, 0::2]) * ref[:, 1::2]
        assert ((o2.float().cpu() - want2).abs().max() / want2.abs().max()) < 6e-3
        # fp32 logits-style output
        o3 = torch.empty(B, N, dtype=torch.float32, device="cuda")
        G.splitk_reduce(ws, o3, bias_along_m=True, ld_m=1, ld_n=N)
        assert ((o3.cpu() - ref).abs().max() / ref.abs().max()) < 2e-5


def test_cluster_reduce_norm_matches_single_cta(G):
    """The 8-CTA cluster reduce+residual+RMSNorm (N >= 1024) against a torch restatement."""
    B, N, S = 16, 4096, 13
    ws = rnd(S, B, N, seed=11).cuda()
    x = rnd(B, N, seed=12).bfloat16().cuda()
    w = (1 + 0.1 * rnd(N, seed=13)).cuda()
    y = torch.empty_like(x)
    x0 = x.clone()
    G.decode_reduce_norm(ws, x, w, y, 1e-5, pdl=False)
    acc = torch.zeros(B, N, device="cuda")
    for si in range(S):            # same summation order as the kernel
        acc = acc + ws[si]
    h = (acc + x0.float()).bfloat16()
    assert torch.equal(x, h)                                       # residual stream: exact
    hf = h.float()
    want = w * (hf * torch.rsqrt(hf.pow(2).mean(-1, keepdim=True) + 1e-5)).bfloat16().float()
    assert ((y.float() - want).abs().max() / want.abs().max()).item() < 8e-3


@pytest.mark.parametrize("B,V,S", [(16, 32114, 8), (3, 1000, 1), (5, 40, 11)])
def test_head_tail_kernel_equals_reduce_argmax_advance(G, B, V, S):
    """groma_decode_head_argmax == groma_splitk_reduce + groma_argmax + groma_decode_advance: logits bit for bit, first-index
    tie-break across thread / CTA boundaries, position bookkeeping."""
    ws = rnd(S, B, V, seed=21).cuda()
    ws[:, 1] = 0.0                                   # one row where every column ties: index 0 wins
    if V > 600:
        ws[:, 0] = 0.0
        ws[0, 0, [7, 513, V - 1]] = 50.0             # equal maxima in different threads and different cluster ranks
        ws[0, 2, V - 1] = 60.0                       # maximum in the last (short) slice
    want = torch.empty(B, V, device="cuda")
    G.splitk_reduce(ws, want)
    ids0 = G.argmax(want)
    logits = torch.empty(B, V, device="cuda")
    ids = torch.full((B,), -1, dtype=torch.int64, device="cuda")
    pos = torch.tensor([41], dtype=torch.int32, device="cuda")
    kvl = torch.arange(B, dtype=torch.int32, device="cuda") + 40
    G.decode_head_argmax(ws, logits, ids, pos, kvl, pdl=False)
    assert torch.equal(logits, want)
    assert torch.equal(ids, ids0) and torch.equal(ids.cpu(), want.cpu().argmax(-1))
    assert ids[1].item() == 0
    if V > 600:
        assert ids[0].item() == 7 and ids[2].item() == V - 1
    assert pos.item() == 42 and torch.equal(kvl.cpu(), torch.arange(B, dtype=torch.int32) + 41)


def test_fused_decode_step_is_bit_identical_to_unfused():
    """The fused reduce epilogues + programmatic dependent launch must not change a single bit of the decode logits."""
    from groma.model.groma import GromaConfig, GromaModel
    from groma_b200.config import SyntheticTokenizer, tiny_config
    from groma_b200.synth import make_state_dict
    cfg = tiny_config(box_score_thres=0.0)
    tok = SyntheticTokenizer(cfg.vocab)
    m = GromaModel(GromaConfig.from_path_config(cfg), state_dict=make_state_dict(cfg, seed=0), path_config=cfg)
    m.init_special_token_id(tok)
    g = torch.Generator().manual_seed(3)
    images = torch.randn(2, 3, 448, 448, generator=g)
    ids = torch.randint(10, cfg.vocab, (2, 16), generator=g)
    ids[:, 2] = tok.map["<image>"]; ids[:, 9] = tok.map["<region>"]
    boxes = [torch.rand(4, 4, generator=g) * 0.6 + 0.2, torch.rand(6, 4, generator=g) * 0.6 + 0.2]
    runs = {}
    for fused, pdl, graph in [(False, False, False), (True, False, False), (True, True, False), (True, True, True)]:
        m.engine.fused_decode, m.engine.use_pdl, m.use_cuda_graph = fused, pdl, graph
        m._graph = None
        out = m.generate(ids.clone().cuda(), images=images.cuda(), max_new_tokens=6, return_dict_in_generate=True,
                         _selected_override=boxes, _keep_logits=True)
        runs[(fused, pdl, graph)] = (out.sequences.cpu(), torch.stack([x.cpu() for x in m._step_logits], 1))
    base_seq, base_lg = runs[(False, False, False)]
    for k, (seq, lg) in runs.items():
        assert torch.equal(seq, base_seq), k
        assert torch.equal(lg, base_lg), k    # tiny model: N=256 < 1024 keeps the single-CTA reduce -> bit-identical
    # all fused variants agree with each other bit for bit (same kernels; PDL / graph only change scheduling)
    assert torch.equal(runs[(True, False, False)][1], runs[(True, True, True)][1])


@pytest.mark.parametrize("ragged", [False, True])
def test_rope_attention_fusion_is_bit_identical(G, ragged):
    """groma_decode_rope_attention == groma_decode_reduce_rope_kv followed by groma_decode_attention: attention output and the
    appended K/V rows, bit for bit (head_dim 128, the Groma-7B shape; the miniature model's decode uses head_dim 32)."""
    torch.manual_seed(5)
    B, H, D, cap, S, pos = 5, 4, 128, 300, 3, 257
    dev = "cuda"
    ws = torch.randn(S, B, 3 * H * D, device=dev)
    kc0 = torch.randn(B, H, cap, D, device=dev).bfloat16()
    vc0 = torch.randn(B, H, cap, D, device=dev).bfloat16()
    ang = torch.rand(cap, D // 2, device=dev) * 6.28
    cos_t, sin_t = ang.cos().contiguous(), ang.sin().contiguous()
    pos_t = torch.tensor([pos], dtype=torch.int32, device=dev)
    kv = [pos + 1] * B
    if ragged:
        kv = [pos + 1, 17, pos, 1, 130]          # rows whose visible range does not include the appended position
    kv_len = torch.tensor(kv, dtype=torch.int32, device=dev)
    scale = 1.0 / math.sqrt(D)
    k1, v1 = kc0.clone(), vc0.clone()
    q = torch.empty(B, H * D, device=dev, dtype=torch.bfloat16)
    a1 = torch.empty(B, H * D, device=dev, dtype=torch.bfloat16)
    G.decode_reduce_rope_kv(ws, q, k1, v1, cos_t, sin_t, pos_t, H, D, pdl=False)
    G.decode_attention(q, k1, v1, kv_len, scale, a1)
    k2, v2 = kc0.clone(), vc0.clone()
    a2 = torch.empty_like(a1)
    G.decode_rope_attention(ws, k2, v2, kv_len, pos_t, cos_t, sin_t, scale, a2, pdl=False)
    torch.cuda.synchronize()
    assert torch.equal(k1, k2) and torch.equal(v1, v2)
    assert not torch.equal(k1[:, :, pos], kc0[:, :, pos])          # the row really was appended
    assert torch.equal(a1, a2)
