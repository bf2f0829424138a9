#!/usr/bin/env python
"""Benchmark of the Groma-7B forward hot path on B200 (BASELINE.json metric: images/sec, 448px prefill + 128-token
greedy decode).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle) on the host cores
  python bench.py ... --dump-outputs DIR                   # also write what the last timed step returned to DIR/<name>.npy

One "step" = one GromaModel.generate() over a batch of 16 synthetic 448x448 images + 512-token prompts per GPU
(BASELINE.json configs[3]; weak scaling = configs[4]), random-init Groma-7B weights (no network for checkpoints).
`value` times the step with inputs resident in HBM; `e2e` times the same public-API call with HOST (pinned) inputs:
H2D of images/ids and D2H of the generated sequences are inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="images per GPU")
    ap.add_argument("--prompt", type=int, default=512)
    ap.add_argument("--new", type=int, default=128)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-check", action="store_true",
                    help="skip the full-size GPU-vs-oracle parity check that rides in the JSON line as `parity_check` (N=1 only)")
    ap.add_argument("--tiny", action="store_true", help="debug: miniature model")
    ap.add_argument("--profile", action="store_true", help="print a per-stage CUDA-event breakdown of one step to stderr")
    ap.add_argument("--ncu-range", action="store_true",
                    help="wrap ONE extra step in cudaProfilerStart/Stop (use with ncu --profile-from-start off --graph-profiling node)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what generate() returned in the last one to DIR/<name>.npy (float32 / "
                         "float64; outputs larger than 2^21 elements as a fixed seeded sample), for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


METRIC = "images/sec Groma-7B 448px prefill+128-tok decode"


DUMP_SAMPLE = 1 << 21          # elements kept of an output larger than this (8 MB in float32)


def _dump_sample(t: torch.Tensor, n: int, seed: int) -> torch.Tensor:
    """`t` whole if it has at most `n` elements, else `n` of its elements at flat indices drawn from `seed` (sorted): the same
    indices for the same shape, so two runs compare element for element."""
    if t.numel() <= n:
        return t
    idx = torch.randint(t.numel(), (n,), generator=torch.Generator().manual_seed(seed)).sort().values.to(t.device)
    return t[torch.unravel_index(idx, t.shape)]


def dump_outputs(out_dir: str, seq: torch.Tensor, out) -> dict:
    """What GromaModel.generate() returned to its caller: the sequences (token ids, exact in float64), the selected boxes of
    every image, the image and region features and the KV cache.  Returns {name: bytes written}."""
    import numpy as np
    vis = out.hidden_states[0][-1]
    kv = [t for layer in out.past_key_values for t in layer]          # 2 x layers tensors [B, heads, ctx, head_dim]
    arrays = {
        "sequences": seq.double(),
        "pred_boxes": torch.cat(vis["pred_boxes"]).float(),
        "regions_per_image": torch.tensor([len(b) for b in vis["pred_boxes"]], dtype=torch.float64),
        "image_features": _dump_sample(vis["image_features"], DUMP_SAMPLE, 1).float(),
        "region_features": _dump_sample(vis["region_features"], DUMP_SAMPLE, 2).float(),
        "past_key_values": torch.stack([_dump_sample(t, DUMP_SAMPLE // len(kv), 3 + i) for i, t in enumerate(kv)]).float(),
    }
    os.makedirs(out_dir, exist_ok=True)
    written = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a)
        written[name] = a.nbytes
    assert sum(written.values()) <= 64 << 20, written
    return written


def make_inputs(cfg, B, T_text, seed, tok):
    g = torch.Generator().manual_seed(seed)
    images = torch.randn(B, 3, cfg.image_size, cfg.image_size, generator=g)
    ids = torch.randint(1000 if cfg.vocab > 2000 else 10, cfg.vocab, (B, T_text), generator=g)
    ids[:, 4] = tok.map["<image>"]
    ids[:, T_text // 2] = tok.map["<region>"]
    return images, ids


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = sorted(float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 7 and r[3 + k].lower().startswith("active") for r in self.rows)]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------ reference arm (CPU)
def usable_cores() -> int:
    """Cores this process may actually use: affinity mask capped by the cgroup CPU quota (the GPU boxes expose 128 logical
    CPUs under a 16-CPU quota; 128 threads there run ~20x slower than 16)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(p) + 0.5)))
    except Exception:
        pass
    return n


def cpu_reference(cfg, tok, T_text, n_new_full, sd_cpu, decode_steps=2):
    """The reference's CPU path = the fp32 oracle (oracle/groma_oracle.py; the reference itself cannot be imported in
    this image, SURVEY.md T12).  Bounded sample: ONE image -- vision + proposer + region encoder + prefill timed in full,
    `decode_steps` decode steps timed and extrapolated to the 128-token decode of the metric."""
    from oracle.groma_oracle import Oracle
    cores = usable_cores()
    torch.set_num_threads(cores)
    o = Oracle(cfg, sd_cpu, "fp32")
    o.init_special_token_id(tok)
    images, ids = make_inputs(cfg, 1, T_text, 1234, tok)
    torch.manual_seed(0)
    t0 = time.time()
    out = o.forward_prefill(ids.clone(), images)
    t1 = time.time()
    nxt, kv = out["logits"][:, -1].argmax(-1), out["kv"]
    for _ in range(decode_steps):
        lg, kv = o.forward_decode(nxt[:, None], kv)
        nxt = lg[:, -1].argmax(-1)
    t2 = time.time()
    per_img = (t1 - t0) + (t2 - t1) / decode_steps * (n_new_full - 1)
    return {"value": 1.0 / per_img, "unit": "images/sec", "cores": cores, "kind": "port",
            "sample": f"1 image, {T_text}-token prompt, R={len(out['selected_boxes'][0])}: vision+prefill {t1 - t0:.1f}s measured, "
                      f"{decode_steps} decode steps measured ({(t2 - t1) / decode_steps:.2f}s/step) extrapolated to {n_new_full - 1}",
            "prefill_s": t1 - t0, "decode_step_s": (t2 - t1) / decode_steps}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    from groma_b200.config import PathConfig, SyntheticTokenizer, tiny_config
    cfg = tiny_config(box_score_thres=0.0) if args.tiny else PathConfig(box_score_thres=0.0)
    tok = SyntheticTokenizer(cfg.vocab)
    workload = {"workload": f"Groma-7B e2e: batch {args.batch}/GPU, 448x448 synthetic images, {args.prompt}-token prompts, "
                            f"prefill (256 image + 2R region + text tokens, R<=100 from NMS at score_thres 0) + {args.new}-token greedy decode "
                            f"(BASELINE.json configs[3]; configs[4] at 8 GPUs)",
                "global_batch": args.batch * world, "prompt_tokens": args.prompt, "new_tokens": args.new,
                "parallelism": f"dp{world} (image-batch shards, weights replicated)",
                "l2": "every step streams 14.8 GB of weights (>> 126 MB L2): inputs larger than L2, no explicit flush"}

    if args.impl == "reference":
        if rank != 0:
            return
        from groma_b200.synth import make_state_dict
        sd = make_state_dict(cfg, seed=0, perturb_norms=False)
        cb = cpu_reference(cfg, tok, args.prompt, args.new, sd)
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "images/sec", "n_gpus": args.gpus, "steps": 1,
                "warmup": 0, "ms_per_step": 1000.0 / cb["value"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": workload, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    assert torch.cuda.is_available(), "bench.py needs a GPU (the B200 path has no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        import datetime
        import torch.distributed as dist
        dist.init_process_group("nccl", timeout=datetime.timedelta(seconds=180))   # fail fast instead of a 10-minute watchdog
    from groma_b200 import ops as G
    from groma_b200.synth import make_state_dict
    from groma.model.groma import GromaConfig, GromaModel

    sd = make_state_dict(cfg, seed=0, perturb_norms=False, dtype=torch.bfloat16, device="cuda")
    model = GromaModel(GromaConfig.from_path_config(cfg), state_dict=sd, path_config=cfg)
    model.init_special_token_id(tok)
    sd_for_cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sd_for_cpu = sd
    else:
        del sd
    torch.cuda.empty_cache()

    B = args.batch
    images_h, ids_h = make_inputs(cfg, B, args.prompt, 1000 + rank, tok)   # each rank draws its own shard of the global batch
    images_h, ids_h = images_h.pin_memory(), ids_h.pin_memory()
    images_d, ids_d = images_h.cuda(), ids_h.cuda()
    realised = {}

    def step(host_inputs: bool):
        torch.manual_seed(0)      # same CPU generator state on every rank: randperm draws are replayed in global image order
        if host_inputs:
            img = images_h.cuda(non_blocking=True)
            ids = ids_h.cuda(non_blocking=True)
        else:
            img, ids = images_d, ids_d.clone()
        out = model.generate(ids, images=img, max_new_tokens=args.new, return_dict_in_generate=True, output_hidden_states=True)
        seq = out.sequences
        boxes = out.hidden_states[0][-1]["pred_boxes"]
        if world > 1:
            # the path's only exchange step (SURVEY section 8e): fixed-shape all-gather of ids + boxes over NCCL
            from groma_b200.dist import gather_outputs
            seq, _, _ = gather_outputs(seq, boxes, cfg.max_region_num)
        if host_inputs:
            seq = seq.cpu()
        realised["R"] = [len(b) for b in boxes]
        realised["T"] = model._path_cfg.grid ** 2 // 4 + args.prompt - 2 + 2 * max(realised["R"])
        realised["outputs"] = (seq, out)
        return seq

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(host_inputs: bool, K: int):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = G.LAUNCHES
        s.record()
        for _ in range(K):
            step(host_inputs)
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device="cuda")
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), G.LAUNCHES - l0

    for _ in range(max(args.warmup, 1)):
        step(True)
    if args.profile:            # every rank runs the step (it contains collectives); rank 0 prints
        model.profile = []
        step(False)
        torch.cuda.synchronize()
        marks, model.profile = model.profile, None
        for (n0, e0), (n1, e1) in zip(marks[:-1], marks[1:]):
            if rank == 0:
                print(f"[profile] {n1:>16s}: {e0.elapsed_time(e1):9.3f} ms", file=sys.stderr)
        if rank == 0:
            print(f"[profile] {'total':>16s}: {marks[0][1].elapsed_time(marks[-1][1]):9.3f} ms", file=sys.stderr)
    if args.ncu_range:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step(False)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_dev, launches_dev = timed(False, args.steps)
    ms_e2e, _ = timed(True, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    dumped = None
    if args.dump_outputs and rank == 0:     # before the roofline below, which overwrites the KV cache
        dumped = dump_outputs(args.dump_outputs, *realised.pop("outputs"))
    realised.pop("outputs", None)

    # kernels launched inside one timed step: C-ABI launches made eagerly + kernels replayed from the decode graph
    graph_kernels = getattr(model, "_graph_kernels", 0)
    replays = max(args.new - 2, 0)
    gpu_launches = launches_dev // max(args.steps, 1) + replays * graph_kernels

    # ---- roofline of the dominant kernel: the swap-AB tcgen05 GEMM that streams the LLaMA weights during decode
    roof = decode_gemm_roofline(model, B, args, step)   # all ranks: the step contains collectives; rank 0 reports its own

    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    n_img = B * world * args.steps
    value = n_img / (ms_dev / 1000.0)
    e2e_v = n_img / (ms_e2e / 1000.0)
    line = {"metric": METRIC, "value": value, "unit": "images/sec", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic (randn images, uniform random prompt ids, random-init weights of the Groma-7B architecture)",
            "config": dict(workload, realised_regions_per_image=realised.get("R"), prefill_tokens=realised.get("T")),
            "clocks": clocks,
            "e2e": {"value": e2e_v, "unit": "images/sec", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": int(images_h.numel() * 4 + ids_h.numel() * 8),
                    "d2h_bytes_per_step": int(B * world * (args.prompt + args.new) * 8)},
            "gpu_launches": int(gpu_launches), "roofline": roof}
    if dumped is not None:
        line["dumped_outputs"] = {"dir": args.dump_outputs, "bytes": dumped}
    if sd_for_cpu is not None:
        sd_cpu = {k: v.float().cpu() for k, v in sd_for_cpu.items()}
        del sd_for_cpu
        line["cpu_baseline"] = cpu_reference(cfg, tok, args.prompt, args.new, sd_cpu)
        if not args.no_check:
            line["parity_check"] = parity_check(model, cfg, sd_cpu, tok, args)
    else:
        line["cpu_baseline"] = None
    print(json.dumps(line))


def parity_check(model, cfg, sd_cpu, tok, args):
    """Not timed, not part of `value`: the SAME weights the timed steps ran on, one image + one prompt of the benchmark's
    length through the GPU path and through the CPU oracle (the checker), stage by stage -- tests/fullsize.py.  Keys:
    every `*_nrel` / `*_max_abs` distance, the exactness flags of the integer stages, `violations` (bars of
    tests/test_fullsize_gpu.py that are not met; empty = green)."""
    try:
        from tests.fullsize import BARS, run_fullsize_check, verdict
        res = run_fullsize_check(model, cfg, sd_cpu, tok, n_text=args.prompt, n_new=8, log=lambda m: print(m, file=sys.stderr))
        res["violations"] = verdict(res)
        res["bars"] = BARS
        return res
    except Exception as e:   # the benchmark line must survive a checker failure
        import traceback
        traceback.print_exc(file=sys.stderr)
        return {"error": f"{type(e).__name__}: {e}"}


def _graph_of(fn):
    g = torch.cuda.CUDAGraph()
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        fn()
        with torch.cuda.graph(g, stream=st, capture_error_mode="thread_local"):
            fn()
    torch.cuda.current_stream().wait_stream(st)
    return g


def _time_graph(g, reps=10, before=None):
    for _ in range(3):
        if before:
            before()
        g.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = 0.0
    for _ in range(reps):
        if before:
            before()
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        ms += e0.elapsed_time(e1)
    return ms / reps


def _traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of this round
    (profiles/r02_dram_traffic.json, written by tools/ncu_summary.py), or None when the kernel was not captured."""
    path = os.path.join(ROOT, "profiles", "r02_dram_traffic.json")
    if not os.path.exists(path):
        return None
    return json.load(open(path)).get(kernel_key)


def decode_gemm_roofline(model, B, args, step):
    """Roofline of the dominant kernel of the step, measured live with CUDA events on the launching stream.

    Decode is ~2/3 of the step and HBM-bound.  Algorithmic bytes are SURVEY.md section 8(d)'s: the bf16 weights every decode step
    has to read (13.22 GB: 32 layers x (qkv, o, gate/up, down) + both heads) and, for kernels that also stream the cache, the K/V
    rows (B x ctx x 0.5 MiB) -- activations, split-K partials and flags are implementation traffic and are NOT counted.
      * persistent kernel (default when supported): ONE launch per step = `decode_step_megakernel`; its duration is a graph replay
        of (flag reset + kernel) at the benchmark's mid-decode context.
      * multi-kernel step: the swap-AB tcgen05 GEMM (129 launches per step, weights only) in a GEMM-only graph with the step's
        split-K factors and PDL attributes, plus `decode_attention_tma_kernel` (32 launches, K/V only) as the second entry."""
    eng = model.engine
    cfg = eng.cfg
    from groma_b200 import ops as G
    d = eng._decode_buffers(B)
    peak, how = peaks()
    Hd, I, V, L = cfg.llm_hidden, cfg.llm_inter, cfg.vocab + cfg.num_new_token, cfg.llm_layers
    wbytes = L * (4 * Hd * Hd + 3 * Hd * I) * 2 + V * Hd * 2
    ctx = int(eng.past) - args.new // 2 if getattr(eng, "past", None) else 1030        # mid-decode context of the timed steps
    ctx = max(ctx, 1)
    kvbytes = L * 2 * B * (ctx + 1) * Hd * 2
    note = ("the 6.58 TB/s peak is a copy (read+write); a read-only stream reaches 7.35 TB/s on this part (tools/cu/read_bw.cu, LDG.128 or "
            "1-D bulk TMA), so frac vs read-only would be achieved/7350")

    def reset():
        d["pos"].fill_(ctx)
        d["kv_len"].fill_(ctx + 1)

    entries = []
    if eng.use_megakernel and eng.mega_supported(B):
        reset()
        ms = _time_graph(_graph_of(lambda: eng.decode_step_mega(B)), reps=20, before=reset)
        eng.check_decode_status()
        ach = (wbytes + kvbytes) / (ms / 1000.0) / 1e9
        entries.append({"kernel": "decode_step_megakernel (one persistent launch per decode step: 32 layers + heads + argmax)", "bound": "hbm",
                        "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": _traffic("decode_step_megakernel"),
                        "peak_source": how, "launches_timed": 20, "avg_launch_us": ms * 1000.0,
                        "algorithmic_bytes_per_launch": wbytes + kvbytes, "algorithmic_bytes": {"weights": wbytes, "kv_cache": kvbytes, "ctx": ctx},
                        "read_only_ceiling_note": note})
    sp = eng._decode_splits()
    names = []
    for i in range(L):
        names += [(f"llm.{i}.qkv.w", sp["qkv"], "y"), (f"llm.{i}.o.w", sp["o"], "q"), (f"llm.{i}.gu.w", sp["gu"], "y"), (f"llm.{i}.down.w", sp["down"], "gu")]
    names.append(("head.w", sp["head"], "y"))

    def gemms():
        for wname, split, src in names:
            W = eng.w[wname]
            ws = d["ws"][: split * W.shape[0] * B].view(split, B, W.shape[0])
            G.gemm_swap_ab(d[src], W, ws, split_k=split, pdl=eng.use_pdl, transposed=True)

    ms = _time_graph(_graph_of(gemms))
    ach = wbytes / (ms / 1000.0) / 1e9
    entries.append({"kernel": "gemm_bf16_tcgen05_kernel<16> (swap-AB weight-streaming GEMM of the multi-kernel decode step; 129 launches per step)",
                    "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": _traffic("gemm_bf16_tcgen05_kernel<16>"), "peak_source": how, "launches_timed": len(names) * 10,
                    "avg_launch_us": ms * 1000.0 / len(names), "algorithmic_bytes_per_launch": wbytes / len(names),
                    "algorithmic_bytes": {"weights": wbytes}, "read_only_ceiling_note": note})
    if cfg.head_dim == 128:
        import math
        reset()

        def attns():
            for i in range(L):
                G.decode_attention(d["q"], eng.kv[i, 0], eng.kv[i, 1], d["kv_len"], 1.0 / math.sqrt(128), d["a"], pdl=eng.use_pdl)
        ms = _time_graph(_graph_of(attns))
        ach = kvbytes / (ms / 1000.0) / 1e9
        entries.append({"kernel": "decode_attention_tma_kernel<128> (single-query attention over the KV cache; 32 launches per step)", "bound": "hbm",
                        "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": _traffic("decode_attention_tma_kernel"),
                        "peak_source": how, "launches_timed": L * 10, "avg_launch_us": ms * 1000.0 / L, "algorithmic_bytes_per_launch": kvbytes / L,
                        "algorithmic_bytes": {"kv_cache": kvbytes, "ctx": ctx}})
    primary = dict(entries[0])
    primary["other_kernels"] = entries[1:]
    return primary


if __name__ == "__main__":
    main()
