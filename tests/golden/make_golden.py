"""Generates tests/golden/tiny_forward.pt: outputs of the CPU oracle ('bf16' mode, seed 0, tiny_config) for one fixed
2-image batch.  The reference itself cannot be imported in this image (SURVEY.md T12), so these vectors pin the
restatement against silent drift -- and the GPU path (tests/test_golden_gpu.py) against the restatement -- rather
than against the reference.   python -m tests.golden.make_golden

The oracle runs under CANONICAL_CPU_ENV so that the fixture is bit-for-bit what any x86-64 machine computes: with the
default settings the fp32 sums differ with the CPU's vector ISA and thread count, and the bf16 rounding points turn such
last-bit differences into different greedy tokens or NMS orders wherever two candidates are nearly tied.
"""
import os
import subprocess
import sys

import torch

from oracle.config import SyntheticTokenizer, tiny_config
from oracle.groma_oracle import Oracle
from oracle.weights import make_state_dict

HERE = os.path.dirname(os.path.abspath(__file__))
# one thread, ATen's portable (non-AVX) kernels, oneDNN at its baseline ISA, MKL in conditional-numerical-reproducibility
# mode; all are read when torch loads, hence the child process of run_canonical()
CANONICAL_CPU_ENV = {"ATEN_CPU_CAPABILITY": "default", "ONEDNN_MAX_CPU_ISA": "SSE41", "MKL_CBWR": "COMPATIBLE",
                     "OMP_NUM_THREADS": "1", "MKL_NUM_THREADS": "1"}


def inputs():
    cfg = tiny_config(box_score_thres=0.05)
    tok = SyntheticTokenizer(cfg.vocab)
    g = torch.Generator().manual_seed(2024)
    images = torch.randn(2, 3, 448, 448, generator=g)
    ids = torch.randint(10, cfg.vocab, (2, 20), generator=g)
    ids[:, 2] = tok.map["<image>"]
    ids[:, 11] = tok.map["<region>"]
    ids[0, 16:] = tok.pad_token_id
    return cfg, tok, images, ids


def run_oracle():
    cfg, tok, images, ids = inputs()
    o = Oracle(cfg, make_state_dict(cfg, seed=0), "bf16")
    o.init_special_token_id(tok)
    torch.manual_seed(99)           # the randperm draws of groma.py:275
    out = o.generate(ids.clone(), images, 5)
    return dict(input_ids=out["input_ids"], new_tokens=out["new_tokens"], nms_inds=[torch.from_numpy(x) for x in out["nms_inds"]],
                pred_boxes=out["pred_boxes"], scores=out["scores"], selected_boxes=out["selected_boxes"],
                last_logits=out["logits"][:, -1].clone(), step_logits=out["step_logits"], topk=o.stages["topk"].clone())


def run_canonical(path):
    """run_oracle() in a child process under CANONICAL_CPU_ENV; its outputs are saved to `path` and returned."""
    root = os.path.dirname(os.path.dirname(HERE))
    subprocess.run([sys.executable, "-m", "tests.golden.make_golden", path], cwd=root, env=dict(os.environ, **CANONICAL_CPU_ENV),
                   check=True)
    return torch.load(path)


if __name__ == "__main__":
    if len(sys.argv) > 1:           # the child of run_canonical()
        assert all(os.environ.get(k) == v for k, v in CANONICAL_CPU_ENV.items())
        torch.save(run_oracle(), sys.argv[1])
    else:
        out = run_canonical(os.path.join(HERE, "tiny_forward.pt"))
        print({k: (tuple(v.shape) if hasattr(v, "shape") else len(v)) for k, v in out.items()})
